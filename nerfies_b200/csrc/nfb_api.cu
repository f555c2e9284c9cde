// C ABI of nerfies_b200 (see include/nerfies_b200.h): handle, parameter
// packing, workspace and the launch sequence of NerfModel.__call__.
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <cstdlib>
#include <string>
#include <vector>

#include "../../include/nerfies_b200.h"
#include "common.cuh"
#include "nfb_handle.h"
#include "field_simt.cuh"
#include "ray_kernels.cuh"
#include "camera_kernels.cuh"
#include "tc_common.cuh"
#include "tc_selftest.cuh"
#include "tc_selftest2.cuh"
#include "tc_selftest3.cuh"
#ifdef NFB_WITH_TC
#include "field_tc.cuh"
#include "field_tc3.cuh"
#endif

namespace {

using nfb::FieldProgram;
using nfb::Net;
using nfb::Step;

struct Builder {
  nfb_handle* h;
  long long off = 0;  // running float offset in the packed buffer

  long long alloc(long long n) {
    long long o = off;
    off += (n + 3) / 4 * 4;  // keep 16-byte alignment for cp.async
    return o;
  }

  // Adds one Dense layer made of `nparts` reference tensors side by side in N
  // (the SE(3) w and v heads are fused into one N=6 step).
  Step dense(const std::vector<std::string>& names, int k_x, int k_in, int in_off,
             const std::vector<int>& ns, int act, int src, int dst) {
    int n = 0;
    for (int v : ns) n += v;
    Step st{};
    st.k_x = k_x; st.k_in = k_in; st.in_off = in_off;
    st.n = n; st.npad = pad32(n);
    st.act = act; st.src = src; st.dst = dst;
    const int K = k_x + k_in;
    st.w_off = (int)alloc((long long)K * st.npad);
    st.b_off = (int)alloc(st.npad);
    int c = 0;
    for (size_t i = 0; i < names.size(); ++i) {
      h->specs.push_back({names[i] + "/kernel", K, ns[i], st.w_off, st.npad, c, 0});
      h->specs.push_back({names[i] + "/bias", 1, ns[i], st.b_off, st.npad, c, 0});
      c += ns[i];
    }
    return st;
  }
};

int build_mlp(Builder& b, Net& net, const std::string& prefix, int depth, int width,
              unsigned skips, int in_dim, int in_off, int act, int first_src, int first_kx,
              int* cur_buf /* in: buffer holding X (if first_kx>0); out: buffer with result */) {
  // modules.MLP (modules.py:39-62): x = act(Dense([x, inputs] if i in skips else x)).
  int cur = *cur_buf;
  for (int i = 0; i < depth; ++i) {
    const bool skip = (skips >> i) & 1u;
    int k_x, k_in;
    if (i == 0) {
      if (skip) return fail("%s: a skip connection at layer 0 is not supported", prefix.c_str());
      k_x = first_kx; k_in = in_dim;
    } else {
      k_x = width; k_in = skip ? (first_kx + in_dim) : 0;
      if (skip && first_kx) return fail("%s: skip with a non-input first operand unsupported", prefix.c_str());
    }
    const int src = (i == 0) ? first_src : cur;
    int dst = (src == nfb::kB0) ? nfb::kB1 : nfb::kB0;
    if (net.n_steps >= nfb::kMaxSteps) return fail("too many layers");
    net.steps[net.n_steps++] = b.dense({prefix + "/hidden_" + std::to_string(i)}, k_x, k_in,
                                       in_off, {width}, act, src, dst);
    cur = dst;
  }
  *cur_buf = cur;
  return 0;
}

int build_programs(nfb_handle* h) {
  const nfb_config& c = h->cfg;
  Builder b{h};
  const bool use_warp = c.warp_field_type != NFB_WARP_NONE;
  const int G = use_warp ? c.num_warp_features : 0;
  const int A = c.num_appearance_features;
  const int tc = (c.use_appearance_metadata && c.use_trunk_condition) ? A : 0;
  const int ac = (c.use_appearance_metadata && c.use_alpha_condition) ? A : 0;
  int rc = 0;
  if (c.use_viewdirs) rc += 3 + 6 * c.num_nerf_viewdir_freqs;
  rc += ac;  // models.py:206-207: guarded by use_alpha_condition
  if (c.use_camera_metadata) rc += c.num_camera_features;
  const int Dp = 3 + 6 * c.num_nerf_point_freqs;
  const int Dw = 3 + 6 * c.num_warp_freqs + G;
  h->cond_stride = G + tc + ac + rc;
  if (h->cond_stride == 0) h->cond_stride = 1;
  if (Dp + tc + ac + rc > nfb::kMaxIn || (use_warp && Dw > nfb::kMaxIn))
    return fail("input feature block wider than %d", nfb::kMaxIn);
  auto check_width = [&](int w, const char* what) {
    if (w < 1 || w > nfb::kMaxWidth)
      return fail("%s=%d outside [1,%d]", what, w, nfb::kMaxWidth);
    return 0;
  };
  if (check_width(c.nerf_trunk_width, "nerf_trunk_width")) return -1;
  if (c.nerf_rgb_branch_depth > 0 && check_width(c.nerf_rgb_branch_width, "nerf_rgb_branch_width")) return -1;
  if (use_warp && check_width(c.warp_trunk_width, "warp_trunk_width")) return -1;
  if (c.alpha_channels != 1 || c.rgb_channels != 3)
    return fail("alpha_channels/rgb_channels must be 1/3 (volumetric_rendering assumes it)");
  if (c.nerf_trunk_depth < 1) return fail("nerf_trunk_depth must be >= 1");

  // Embedding tables come first in the parameter order (Flax names).
  Net warp{};
  if (use_warp) {
    // metadata encoder of the warp field (warping.py:109-123, 250-260)
    const int enc = c.warp_metadata_encoder;
    if (enc < NFB_WARP_ENC_GLO || enc > NFB_WARP_ENC_BLEND) return fail("bad warp_metadata_encoder");
    if (enc == NFB_WARP_ENC_BLEND && c.warp_field_type != NFB_WARP_TRANSLATION)
      return fail("Unknown metadata encoder type 'blend' for the SE(3) field (warping.py:258-260)");
    if (enc != NFB_WARP_ENC_TIME)
      h->specs.push_back({std::string(enc == NFB_WARP_ENC_GLO ? "warp_field/metadata_encoder" : "warp_field/glo_encoder") +
                          "/embed/embedding", c.num_warp_embeddings, G, 0, G, 0, 1});
    if (enc != NFB_WARP_ENC_GLO) {
      // modules.TimeEncoder (modules.py:297-322): depth 6, width 64, skips (4,), output = G features
      const int F = c.time_encoder_num_freqs;
      if (F < 0 || 1 + 2 * F > nfb::kTimeMaxIn) return fail("metadata_encoder_num_freqs=%d unsupported", F);
      const std::string root = enc == NFB_WARP_ENC_TIME ? "warp_field/metadata_encoder/mlp" : "warp_field/time_encoder/mlp";
      int tcur = nfb::kB0;
      Net tn{};
      if (build_mlp(b, tn, root, 6, 64, 1u << 4, 1 + 2 * F, 0, nfb::kRelu, nfb::kB0, 0, &tcur)) return -1;
      tn.steps[tn.n_steps++] = b.dense({root + "/logit"}, 64, 0, 0, {G}, nfb::kNone, tcur, nfb::kOut0);
      h->time_net = tn;
    }
    if (c.warp_field_type != NFB_WARP_SE3 && (c.warp_use_pivot || c.warp_use_translation))
      return fail("use_pivot / use_translation are SE3Field arguments (warping.py:242-243)");
    int cur = nfb::kB0;
    const bool se3 = c.warp_field_type == NFB_WARP_SE3;
    const std::string mlp_name = se3 ? "warp_field/trunk" : "warp_field/mlp";
    if (c.warp_trunk_depth < 1) return fail("warp trunk depth must be >= 1");
    if (build_mlp(b, warp, mlp_name, c.warp_trunk_depth, c.warp_trunk_width, c.warp_skips_mask,
                  Dw, 0, nfb::kRelu, nfb::kB0, 0, &cur)) return -1;
    if (se3) {
      // heads side by side in N: [w v (p) (t)] (warping.py:269-303)
      std::vector<std::string> names = {"warp_field/branches_w/logit", "warp_field/branches_v/logit"};
      std::vector<int> ns = {3, 3};
      if (c.warp_use_pivot) { names.push_back("warp_field/branches_p/logit"); ns.push_back(3); }
      if (c.warp_use_translation) { names.push_back("warp_field/branches_t/logit"); ns.push_back(3); }
      warp.steps[warp.n_steps++] = b.dense(names, c.warp_trunk_width, 0, 0, ns, nfb::kNone, cur, nfb::kOut0);
    } else {
      warp.steps[warp.n_steps++] = b.dense({"warp_field/mlp/logit"}, c.warp_trunk_width, 0, 0,
                                           {3}, nfb::kNone, cur, nfb::kOut0);
    }
  }
  if (c.use_appearance_metadata)
    h->specs.push_back({"appearance_encoder/embed/embedding", c.num_appearance_embeddings, A, 0, A, 0, 2});
  if (c.use_camera_metadata)
    h->specs.push_back({"camera_encoder/embed/embedding", c.num_camera_embeddings,
                        c.num_camera_features, 0, c.num_camera_features, 0, 3});

  const int levels = c.num_fine_samples > 0 ? 2 : 1;
  for (int lv = 0; lv < levels; ++lv) {
    const std::string root = lv == 0 ? "nerf_mlps_coarse" : "nerf_mlps_fine";
    Net nerf{};
    const int W = c.nerf_trunk_width;
    int cur = nfb::kB0;
    if (build_mlp(b, nerf, root + "/MLP_0", c.nerf_trunk_depth, W, c.nerf_skips_mask, Dp + tc, 0,
                  c.activation, nfb::kB0, 0, &cur)) return -1;
    const int P = cur;
    const int Q = (P == nfb::kB0) ? nfb::kB1 : nfb::kB0;
    const bool has_cond = ac > 0 || rc > 0;
    // Parameter order follows the Flax tree: MLP_0, bottleneck, MLP_1 (rgb), MLP_2 (alpha);
    // execution order is bottleneck, alpha, rgb (alpha must read the trunk output
    // before the rgb branch reuses that buffer).  Specs are re-sorted below.
    const size_t spec_mark = h->specs.size();
    if (has_cond)
      nerf.steps[nerf.n_steps++] = b.dense({root + "/bottleneck"}, W, 0, 0, {W}, nfb::kNone, P, Q);
    // alpha branch (depth 0: logit only), modules.py:152-157.
    const size_t alpha_mark = h->specs.size();
    if (ac > 0)
      nerf.steps[nerf.n_steps++] = b.dense({root + "/MLP_2/logit"}, W, ac, Dp + tc, {1}, nfb::kNone, Q, nfb::kOut0);
    else
      nerf.steps[nerf.n_steps++] = b.dense({root + "/MLP_2/logit"}, W, 0, 0, {1}, nfb::kNone, P, nfb::kOut0);
    const size_t rgb_mark = h->specs.size();
    // rgb branch, modules.py:159-164.
    int rsrc = (rc > 0) ? Q : P;
    int kx = W;
    int kin = rc, inoff = Dp + tc + ac;
    for (int i = 0; i < c.nerf_rgb_branch_depth; ++i) {
      const int dst = (rsrc == nfb::kB0) ? nfb::kB1 : nfb::kB0;
      if (nerf.n_steps >= nfb::kMaxSteps - 1) return fail("too many layers");
      nerf.steps[nerf.n_steps++] = b.dense({root + "/MLP_1/hidden_" + std::to_string(i)}, kx, kin,
                                           inoff, {c.nerf_rgb_branch_width}, c.activation, rsrc, dst);
      rsrc = dst; kx = c.nerf_rgb_branch_width; kin = 0;
    }
    nerf.steps[nerf.n_steps++] = b.dense({root + "/MLP_1/logit"}, kx, kin, inoff, {3}, nfb::kNone, rsrc, nfb::kOut1);
    // Re-order specs to the Flax order: bottleneck, MLP_1..., MLP_2.
    std::vector<ParamSpec> bott(h->specs.begin() + spec_mark, h->specs.begin() + alpha_mark);
    std::vector<ParamSpec> alpha(h->specs.begin() + alpha_mark, h->specs.begin() + rgb_mark);
    std::vector<ParamSpec> rgb(h->specs.begin() + rgb_mark, h->specs.end());
    h->specs.resize(spec_mark);
    h->specs.insert(h->specs.end(), bott.begin(), bott.end());
    h->specs.insert(h->specs.end(), rgb.begin(), rgb.end());
    h->specs.insert(h->specs.end(), alpha.begin(), alpha.end());

    FieldProgram& p = h->prog[lv];
    memset(&p, 0, sizeof(p));
    p.warp = warp;
    p.nerf = nerf;
    p.warp_type = c.warp_field_type;
    p.warp_pivot = use_warp && c.warp_use_pivot; p.warp_trans = use_warp && c.warp_use_translation;
    p.Fw = c.num_warp_freqs; p.G = G; p.Dw = Dw;
    p.Fp = c.num_nerf_point_freqs; p.Dp = Dp;
    p.tc = tc; p.ac = ac; p.rc = rc;
    p.cond_stride = h->cond_stride;
    p.hidden_act = c.activation; p.sigma_act = c.sigma_activation;
    p.alpha_slot = nfb::kOut0; p.rgb_slot = nfb::kOut1;
  }
  if (levels == 1) h->prog[1] = h->prog[0];
  h->packed_floats = b.off;
  return 0;
}

// Host tables exactly as the reference builds them (float32 arithmetic).
void linspace01(int n, std::vector<float>& t) {
  t.resize(n);
  const double step = n > 1 ? 1.0 / (n - 1) : 0.0;
  for (int i = 0; i < n; ++i) t[i] = (float)(i * step);
  if (n > 1) t[n - 1] = 1.0f;
}

int upload(float** dst, const std::vector<float>& v) {
  NFB_CUDA(cudaMalloc(dst, std::max<size_t>(v.size(), 1) * sizeof(float)));
  if (!v.empty()) NFB_CUDA(cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int build_tables(nfb_handle* h) {
  const nfb_config& c = h->cfg;
  const int nc = c.num_coarse_samples;
  std::vector<float> t, z(nc), lower(nc), upper(nc), u;
  linspace01(nc, t);
  const float near_f = c.near_plane, far_f = c.far_plane;
  for (int i = 0; i < nc; ++i) {
    if (!c.use_linear_disparity) {
      // near * (1 - t) + far * t   (model_utils.py:58)
      volatile float a = near_f * (1.f - t[i]);
      volatile float bb = far_f * t[i];
      z[i] = a + bb;
    } else {
      // 1 / (1/near * (1 - t) + 1/far * t)   (model_utils.py:60)
      const float inv_near = (float)(1.0 / (double)near_f), inv_far = (float)(1.0 / (double)far_f);
      volatile float a = inv_near * (1.f - t[i]);
      volatile float bb = inv_far * t[i];
      volatile float s = a + bb;
      z[i] = 1.f / s;
    }
  }
  for (int i = 0; i < nc; ++i) {
    // mids/upper/lower of the stratified branch (model_utils.py:62-64).
    lower[i] = (i == 0) ? z[0] : .5f * (z[i] + z[i - 1]);
    upper[i] = (i == nc - 1) ? z[nc - 1] : .5f * (z[i + 1] + z[i]);
  }
  linspace01(std::max(c.num_fine_samples, 1), u);
  if (upload(&h->d_zlin, z) || upload(&h->d_lower, lower) || upload(&h->d_upper, upper) ||
      upload(&h->d_ulin, u))
    return -1;
  NFB_CUDA(cudaMalloc(&h->d_window, 64 * sizeof(float)));
  return 0;
}

// cosine_easing_window (modules.py:274-294) in float32.
int set_window(nfb_handle* h, float alpha, cudaStream_t stream) {
  if (h->cfg.warp_field_type == NFB_WARP_NONE) return 0;
  if (alpha == h->h_window_alpha) return 0;
  const int F = h->cfg.num_warp_freqs;
  if (F > 64) return fail("num_warp_freqs > 64");
  float w[64];
  const float pi = 3.14159274101257324f;  // float32(np.pi)
  for (int k = 0; k < F; ++k) {
    float x = alpha - (float)k;
    x = fminf(fmaxf(x, 0.f), 1.f);
    volatile float arg = pi * x;
    arg = arg + pi;
    volatile float cv = cosf(arg);
    w[k] = 0.5f * (1.f + cv);
  }
  // Stream-ordered copy from pageable memory: the driver stages it before returning.
  NFB_CUDA(cudaMemcpyAsync(h->d_window, w, F * sizeof(float), cudaMemcpyHostToDevice, stream));
  h->h_window_alpha = alpha;
  return 0;
}

int launch_check(nfb_handle* h, const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail("%s launch failed: %s", what, cudaGetErrorString(e));
  h->launches++;
  return 0;
}

// The TimeEncoder's window: cosine_easing_window(F, alpha) (modules.py:274-294) with alpha =
// time_alpha for 'time' and F for 'blend' (alpha = None, modules.py:318-319, warping.py:131).
void time_window(const nfb_handle* h, float* w) {
  const int F = h->cfg.time_encoder_num_freqs;
  const float alpha = h->cfg.warp_metadata_encoder == NFB_WARP_ENC_TIME ? h->time_alpha : (float)F;
  const float pi = 3.14159274101257324f;
  for (int k = 0; k < F; ++k) {
    float x = alpha - (float)k;
    x = fminf(fmaxf(x, 0.f), 1.f);
    volatile float arg = pi * x;
    arg = arg + pi;
    volatile float cv = cosf(arg);
    w[k] = 0.5f * (1.f + cv);
  }
}

// time_from_ids: `warp_id` holds uint32 ids even for the 'time' encoder, whose TimeEncoder then sees
// float(id) - the background points of the training loss (training.py:121-131).
int run_cond(nfb_handle* h, int B, const float* viewdirs, const unsigned* warp_id,
             const unsigned* app_id, const unsigned* cam_id, cudaStream_t s, bool encoded = false,
             bool time_from_ids = false) {
  const nfb_config& c = h->cfg;
  nfb::CondArgs a{};
  a.viewdirs = viewdirs; a.warp_id = warp_id; a.app_id = app_id; a.cam_id = cam_id;
  a.warp_table = h->d_warp_table; a.app_table = h->d_app_table; a.cam_table = h->d_cam_table;
  a.n_warp = c.num_warp_embeddings; a.n_app = c.num_appearance_embeddings; a.n_cam = c.num_camera_embeddings;
  a.G = h->prog[0].G; a.A = c.num_appearance_features; a.C = c.num_camera_features;
  a.Fv = c.num_nerf_viewdir_freqs;
  a.use_viewdirs = c.use_viewdirs; a.use_app = c.use_appearance_metadata; a.use_cam = c.use_camera_metadata;
  a.use_trunk_c = c.use_trunk_condition; a.use_alpha_c = c.use_alpha_condition;
  a.stride = h->cond_stride; a.cond = h->d_cond; a.num_rays = B;
  a.encoded = encoded;
  if (h->prog[0].G + h->prog[0].tc + h->prog[0].ac + h->prog[0].rc == 0) return 0;
  const long long total = (long long)B * a.stride;
  const int enc = c.warp_field_type != NFB_WARP_NONE ? c.warp_metadata_encoder : NFB_WARP_ENC_GLO;
  if (enc == NFB_WARP_ENC_TIME && !encoded) a.warp_id = nullptr;   // no GLO table; `warp_id` may carry timestamps
  nfb::ray_cond_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(a);
  if (launch_check(h, "ray_cond_kernel")) return -1;
  if (enc != NFB_WARP_ENC_GLO && !encoded && warp_id) {
    // TimeEncoder on metadata['time'] ('time') or on float(id) ('blend'; 'time' with time_from_ids)
    nfb::TimeArgs t{};
    t.params = h->d_packed; t.net = h->time_net;
    t.F = c.time_encoder_num_freqs;
    if (enc == NFB_WARP_ENC_TIME && !time_from_ids) t.time_f = reinterpret_cast<const float*>(warp_id);
    else t.time_id = warp_id;
    time_window(h, t.window);
    t.blend = enc == NFB_WARP_ENC_BLEND; t.time_alpha = h->time_alpha;
    t.cond = h->d_cond; t.stride = h->cond_stride; t.G = h->prog[0].G; t.num_rays = B;
    nfb::time_embed_kernel<<<(B + nfb::kTimeRays - 1) / nfb::kTimeRays, nfb::kTimeThreads, 0, s>>>(t);
    return launch_check(h, "time_embed_kernel");
  }
  return 0;
}

// The fp16x3 kernel can finish a ray on chip (volumetric rendering fused into its rgb epilogue)
// when a ray's samples are whole 128-row tiles.
bool can_fuse_composite(const nfb_handle* h, int S) {
  return h->cfg.precision == NFB_PREC_FP16X3 && S % 128 == 0 && S <= nfb::kMaxSamples;
}

int run_field(nfb_handle* h, int level, long long rows, int S, const float* origins,
              const float* directions, const float* z, float* samples, float* warped,
              bool use_warp, bool warp_only, cudaStream_t s, float* ray_out = nullptr,
              float* ray_weights = nullptr) {
  if (rows == 0) return 0;
  nfb::FieldArgs a{};
  a.ray_out = ray_out; a.ray_weights = ray_weights;
  a.white_bg = h->cfg.use_white_background; a.sample_at_infinity = h->cfg.use_sample_at_infinity;
  a.params = h->d_packed; a.origins = origins; a.directions = directions; a.z_vals = z;
  a.cond = h->d_cond; a.window = h->d_window; a.samples = samples; a.warped = warped;
  a.num_rows = rows; a.samples_per_ray = S; a.use_warp = use_warp; a.warp_only = warp_only;
  a.fast_encode = h->cfg.precision == NFB_PREC_BF16;
  a.trace = h->trace; a.trace_cap = h->trace_cap;
#ifdef NFB_DEV_KNOBS
  {
    // developer builds only: timing experiments whose results are garbage (see FieldArgs::debug)
    static const int dbg = getenv("NFB_DEBUG") ? atoi(getenv("NFB_DEBUG")) : 0;
    a.debug = dbg;
  }
#endif
  a.debug |= h->debug_bits;
  const bool prof = h->profiling && !warp_only;
  if (prof) NFB_CUDA(cudaEventRecord(h->ev[level][0], s));
  int rc;
  if (h->cfg.precision == NFB_PREC_FP32) {
    const long long tiles = (rows + nfb::kTM - 1) / nfb::kTM;
    nfb::field_simt_kernel<<<(unsigned)tiles, nfb::kSimtThreads, nfb::kSimtSmemBytes, s>>>(h->prog[level], a);
    rc = launch_check(h, "field_simt_kernel");
  } else {
#ifdef NFB_WITH_TC
    rc = h->cfg.precision == NFB_PREC_FP16X3 ? nfb::tc3::run_field_x3(h, level, a, s)
                                             : nfb::tc::run_field_tc(h, level, a, s);
#else
    rc = fail("precision %d needs the tcgen05 path, which this build does not contain", h->cfg.precision);
#endif
  }
  if (prof && rc == 0) {
    NFB_CUDA(cudaEventRecord(h->ev[level][1], s));
    h->ev_valid[level] = true;
  }
  return rc;
}

int run_composite(nfb_handle* h, int B, int S, const float* samples, const float* z,
                  const float* directions, float* out, float* weights, cudaStream_t s) {
  if (S > nfb::kMaxSamples) return fail("more than %d samples per ray", nfb::kMaxSamples);
  nfb::CompositeArgs a{};
  a.samples = reinterpret_cast<const float4*>(samples); a.z_vals = z; a.directions = directions;
  a.out = out; a.weights = weights; a.num_rays = B; a.S = S;
  a.white_bg = h->cfg.use_white_background; a.sample_at_infinity = h->cfg.use_sample_at_infinity;
  const int blocks = (B + nfb::kRaysPerBlock - 1) / nfb::kRaysPerBlock;
  const size_t smem = (size_t)nfb::kRaysPerBlock * 3 * S * sizeof(float);
  nfb::composite_kernel<<<blocks, 32 * nfb::kRaysPerBlock, smem, s>>>(a);
  return launch_check(h, "composite_kernel");
}

int run_resample(nfb_handle* h, int B, const float* zc, const float* wc, const float* u_rand,
                 float* zf, cudaStream_t s) {
  const nfb_config& c = h->cfg;
  nfb::ResampleArgs a{};
  a.z_coarse = zc; a.w_coarse = wc; a.u_rand = u_rand; a.u_lin = h->d_ulin; a.z_fine = zf;
  a.num_rays = B; a.nc = c.num_coarse_samples; a.nf = c.num_fine_samples;
  int p = 1;
  while (p < a.nc + a.nf) p <<= 1;
  a.npow2 = p;
  if (a.nc < 3) return fail("hierarchical sampling needs >= 3 coarse samples");
  const int blocks = (B + nfb::kRaysPerBlock - 1) / nfb::kRaysPerBlock;
  const size_t smem = (size_t)nfb::kRaysPerBlock * (2 * a.nc + p) * sizeof(float);
  nfb::resample_kernel<<<blocks, 32 * nfb::kRaysPerBlock, smem, s>>>(a);
  return launch_check(h, "resample_kernel");
}

// The tcgen05 kernels never trap on a protocol error (see tc_common.cuh,
// mbar_wait): they raise a flag in mapped pinned host memory instead.  One int per
// process; every device's copy of the g_nfb_abort symbol points at it.
int* g_abort_host = nullptr;
unsigned long long g_abort_devices = 0;   // devices whose symbol has been set

int ensure_abort_flag() {
#ifdef NFB_WITH_TC
  int dev = 0;
  NFB_CUDA(cudaGetDevice(&dev));
  if (!g_abort_host) {
    NFB_CUDA(cudaHostAlloc(&g_abort_host, sizeof(int), cudaHostAllocMapped | cudaHostAllocPortable));
    *g_abort_host = 0;
  }
  if (dev < 64 && !(g_abort_devices >> dev & 1)) {
    int* dptr = nullptr;
    NFB_CUDA(cudaHostGetDevicePointer(&dptr, g_abort_host, 0));
    NFB_CUDA(cudaMemcpyToSymbol(nfb::tc::g_nfb_abort, &dptr, sizeof(dptr)));
    g_abort_devices |= 1ull << dev;
  }
#endif
  return 0;
}

int abort_check() {
  if (g_abort_host && *reinterpret_cast<volatile int*>(g_abort_host))
    return fail("a tcgen05 kernel aborted: an mbarrier wait timed out (protocol error); its results are invalid "
                "and tensor-core launches are refused until nfb_reset_abort()");
  return 0;
}

// A handle's workspace (cond, z, samples, window table) is shared by its calls: work
// of consecutive calls must be ordered.  Calls on ONE stream are; when the caller
// switches streams the new stream first waits for the previous call's last kernel.
int enter_stream(nfb_handle* h, cudaStream_t s) {
  if (h->last_stream_valid && h->last_stream != s) {
    if (!h->ev_order) NFB_CUDA(cudaEventCreateWithFlags(&h->ev_order, cudaEventDisableTiming));
    NFB_CUDA(cudaEventRecord(h->ev_order, h->last_stream));
    NFB_CUDA(cudaStreamWaitEvent(s, h->ev_order, 0));
  }
  h->last_stream = s; h->last_stream_valid = true;
  return 0;
}

int check_call(nfb_handle* h, int B) {
  if (!h) return fail("null handle");
  if (abort_check()) return -1;
  if (!h->params_set) return fail("nfb_set_params has not been called");
  if (B < 0 || B > h->max_rays) return fail("num_rays=%d outside [0, max_rays=%d]", B, h->max_rays);
  return 0;
}

}  // namespace

extern "C" {

const char* nfb_last_error(void) { return g_error.c_str(); }
const char* nfb_version(void) { return "nerfies_b200 0.1 sm_100a"; }
long long nfb_kernel_launches(const nfb_handle* h) { return h ? h->launches : 0; }

static int launch_camera(const nfb_camera* cam, const float* pixels_in, long long first, long long count,
                         float* origins, float* directions, float* pixels_out, void* stream) {
  if (!cam) return fail("null argument");
  if (count < 0 || first < 0) return fail("negative pixel range");
  if (cam->image_size[0] < 1 || cam->image_size[1] < 1) return fail("image_size must be positive");
  if (!pixels_in && first + count > (long long)cam->image_size[0] * cam->image_size[1])
    return fail("pixel range [%lld, %lld) exceeds the %d x %d frame", first, first + count,
                cam->image_size[0], cam->image_size[1]);
  if (!(cam->focal_length != 0.f) || !(cam->pixel_aspect_ratio != 0.f)) return fail("focal_length and pixel_aspect_ratio must be non-zero");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("no CUDA device: nerfies_b200 has no CPU path");
  if (count == 0) return 0;
  if (!directions) return fail("null argument");
  if ((reinterpret_cast<uintptr_t>(directions) | reinterpret_cast<uintptr_t>(origins)) & 15)
    return fail("origins / directions must be 16-byte aligned");
  if (reinterpret_cast<uintptr_t>(pixels_out) & 7) return fail("pixels must be 8-byte aligned");
  nfb::CameraArgs a{};
  a.cam = *cam; a.pixels_in = pixels_in; a.first = first; a.count = count;
  a.origins = origins; a.directions = directions; a.pixels_out = pixels_out;
  a.has_distortion = 0;                                   // camera.py:201-207
  for (int i = 0; i < 3; ++i) a.has_distortion |= cam->radial_distortion[i] != 0.f;
  for (int i = 0; i < 2; ++i) a.has_distortion |= cam->tangential_distortion[i] != 0.f;
  nfb::camera_rays_kernel<<<(unsigned)((count + 255) / 256), 256, 0, (cudaStream_t)stream>>>(a);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail("camera_rays_kernel launch failed: %s", cudaGetErrorString(e));
  return 0;
}

int nfb_camera_rays(const nfb_camera* cam, long long first_pixel, long long count, float* origins,
                    float* directions, float* pixels, void* stream) {
  return launch_camera(cam, nullptr, first_pixel, count, origins, directions, pixels, stream);
}

int nfb_pixels_to_rays(const nfb_camera* cam, const float* pixels, long long n, float* directions,
                       void* stream) {
  if (!pixels && n > 0) return fail("null argument");
  return launch_camera(cam, pixels, 0, n, nullptr, directions, nullptr, stream);
}

int nfb_set_trace(nfb_handle* h, long long* buffer, int capacity) {
  if (!h) return fail("null handle");
#ifndef NFB_TRACE
  if (buffer) return fail("this build carries no tracer; rebuild with -DNFB_TRACE (tools/build_variant.py)");
#endif
  h->trace = buffer; h->trace_cap = buffer ? capacity : 0;
  return 0;
}

int nfb_debug_provoke_timeout(nfb_handle* h, int enabled) {
  if (!h) return fail("null handle");
  h->debug_bits = enabled ? 8 : 0;
  return 0;
}

int nfb_set_time_alpha(nfb_handle* h, float time_alpha) {
  if (!h) return fail("null handle");
  h->time_alpha = time_alpha;
  return 0;
}

int nfb_set_profiling(nfb_handle* h, int enabled) {
  if (!h) return fail("null handle");
  if (enabled && !h->ev[0][0]) {
    for (int l = 0; l < 2; ++l)
      for (int i = 0; i < 2; ++i) NFB_CUDA(cudaEventCreate(&h->ev[l][i]));
  }
  h->profiling = enabled != 0;
  h->ev_valid[0] = h->ev_valid[1] = false;
  return 0;
}

float nfb_field_time_ms(nfb_handle* h, int level) {
  if (!h || level < 0 || level > 1 || !h->ev_valid[level]) {
    fail("no profiled field launch for level %d", level);
    return -1.f;
  }
  if (cudaEventSynchronize(h->ev[level][1]) != cudaSuccess) { fail("cudaEventSynchronize failed"); return -1.f; }
  float ms = -1.f;
  if (cudaEventElapsedTime(&ms, h->ev[level][0], h->ev[level][1]) != cudaSuccess) { fail("cudaEventElapsedTime failed"); return -1.f; }
  return ms;
}

int nfb_check_abort(void* stream, int synchronize) {
  if (synchronize) NFB_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return abort_check();
}

int nfb_reset_abort(void) {
  // only meaningful once every stream that ran a tensor-core launch has drained
  NFB_CUDA(cudaDeviceSynchronize());
  if (g_abort_host) *reinterpret_cast<volatile int*>(g_abort_host) = 0;
  return 0;
}

int nfb_selftest_gemm(int K, int N, const float* A, const float* W, float* C, void* stream) {
  using namespace nfb::tc;
  if (K < 1 || K > kSelfMaxKb * kBlockK || N < 1 || N > 256) return fail("selftest: K<=320, N<=256");
  if (ensure_abort_flag() || abort_check()) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int nkb = (K + kBlockK - 1) / kBlockK;
  const int n_rows = (N + 15) / 16 * 16;
  std::vector<int> k_map(nkb * kBlockK, -1);
  for (int k = 0; k < K; ++k) k_map[k] = k;
  int* d_map = nullptr;
  __nv_bfloat16* d_w = nullptr;
  NFB_CUDA(cudaMalloc(&d_map, k_map.size() * sizeof(int)));
  NFB_CUDA(cudaMalloc(&d_w, (size_t)nkb * n_rows * kRowBytes));
  NFB_CUDA(cudaMemcpyAsync(d_map, k_map.data(), k_map.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  const long long total = (long long)nkb * n_rows * kBlockK;
  pack_weight_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(W, N, d_map, nkb, N, n_rows, d_w);
  NFB_CUDA(cudaFuncSetAttribute(tc_selftest_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelfSmemBytes));
  tc_selftest_kernel<<<1, 160, kSelfSmemBytes, s>>>(A, K, d_w, nkb, n_rows, N, C);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  cudaFree(d_map);
  cudaFree(d_w);
  if (e != cudaSuccess) return fail("selftest kernel failed: %s", cudaGetErrorString(e));
  return abort_check();
}

int nfb_selftest_gemm2(int K, int N, const float* A, const float* W, float* C, int reps, long long* out,
                       void* stream) {
  using namespace nfb::tc;
  if (K < 1 || K > kSelfMaxKb * kBlockK || (N != 64 && N != 128 && N != 256)) return fail("selftest2: K<=320, N in {64,128,256}");
  if (reps < 1) return fail("selftest2: reps must be >= 1");
  if (ensure_abort_flag() || abort_check()) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int nkb = (K + kBlockK - 1) / kBlockK;
  std::vector<int> k_map(nkb * kBlockK, -1);
  for (int k = 0; k < K; ++k) k_map[k] = k;
  int* d_map = nullptr;
  __nv_bfloat16* d_w = nullptr;
  long long* d_out = nullptr;
  NFB_CUDA(cudaMalloc(&d_map, k_map.size() * sizeof(int)));
  NFB_CUDA(cudaMalloc(&d_w, (size_t)nkb * N * kRowBytes));
  NFB_CUDA(cudaMalloc(&d_out, 2 * sizeof(long long)));
  NFB_CUDA(cudaMemsetAsync(d_out, 0, 2 * sizeof(long long), s));
  NFB_CUDA(cudaMemcpyAsync(d_map, k_map.data(), k_map.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  const long long total = (long long)nkb * N * kBlockK;
  pack_weight_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(W, N, d_map, nkb, N, N, d_w);
  NFB_CUDA(cudaFuncSetAttribute(tc_selftest2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelf2SmemBytes));
  tc_selftest2_kernel<<<2, 160, kSelf2SmemBytes, s>>>(A, K, d_w, nkb, N, C, reps, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  long long h_out[2] = {0, 0};
  if (e == cudaSuccess) e = cudaMemcpy(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost);
  cudaFree(d_map); cudaFree(d_w); cudaFree(d_out);
  if (e != cudaSuccess) return fail("selftest2 kernel failed: %s", cudaGetErrorString(e));
  if (out) { out[0] = h_out[0]; out[1] = h_out[1]; }
  return abort_check();
}

int nfb_selftest_gemm3(int K, int N, const float* A, const float* W, float* C, int reps, long long* out,
                       void* stream) {
  using namespace nfb::tc;
  if (K < 1 || K > kSelf3MaxKb * kBlockK || N < 1 || N > 256) return fail("selftest3: K<=256, N<=256");
  if (reps < 1) return fail("selftest3: reps must be >= 1");
  if ((long long)((K + kBlockK - 1) / kBlockK) * 2 * ((N + 15) / 16 * 16) * kRowBytes > kSelf3WBytes)
    return fail("selftest3: the packed weights must fit %d bytes of shared memory", kSelf3WBytes);
  if (ensure_abort_flag() || abort_check()) return -1;
  cudaStream_t s = (cudaStream_t)stream;
  const int nkb = (K + kBlockK - 1) / kBlockK;
  const int n_rows = (N + 15) / 16 * 16;
  std::vector<int> k_map(nkb * kBlockK, -1);
  for (int k = 0; k < K; ++k) k_map[k] = k;
  int* d_map = nullptr;
  uint8_t* d_w = nullptr;
  long long* d_out = nullptr;
  float* d_max = nullptr;
  NFB_CUDA(cudaMalloc(&d_map, k_map.size() * sizeof(int)));
  NFB_CUDA(cudaMalloc(&d_w, (size_t)nkb * 2 * n_rows * kRowBytes));
  NFB_CUDA(cudaMalloc(&d_out, 2 * sizeof(long long)));
  NFB_CUDA(cudaMalloc(&d_max, sizeof(float)));
  NFB_CUDA(cudaMemsetAsync(d_out, 0, 2 * sizeof(long long), s));
  NFB_CUDA(cudaMemsetAsync(d_max, 0, sizeof(float), s));
  NFB_CUDA(cudaMemcpyAsync(d_map, k_map.data(), k_map.size() * sizeof(int), cudaMemcpyHostToDevice, s));
  absmax_kernel<<<32, 256, 0, s>>>(W, (long long)K * N, d_max);
  const long long total = (long long)nkb * n_rows * kBlockK;
  pack_weight_x3_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(W, N, d_map, nkb, N, n_rows, d_max, d_w);
  float h_max = 0.f;
  NFB_CUDA(cudaMemcpyAsync(&h_max, d_max, sizeof(float), cudaMemcpyDeviceToHost, s));
  NFB_CUDA(cudaStreamSynchronize(s));
  const float inv_scale = 1.f / x3_weight_scale(h_max) / (float)reps;
  NFB_CUDA(cudaFuncSetAttribute(tc_selftest3_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kSelf3SmemBytes));
  tc_selftest3_kernel<<<1, 160, kSelf3SmemBytes, s>>>(A, K, d_w, nkb, n_rows, N, inv_scale, C, reps, d_out);
  cudaError_t e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaStreamSynchronize(s);
  long long h_out[2] = {0, 0};
  if (e == cudaSuccess) e = cudaMemcpy(h_out, d_out, sizeof(h_out), cudaMemcpyDeviceToHost);
  cudaFree(d_map); cudaFree(d_w); cudaFree(d_out); cudaFree(d_max);
  if (e != cudaSuccess) return fail("selftest3 kernel failed: %s", cudaGetErrorString(e));
  if (out) { out[0] = h_out[0]; out[1] = h_out[1]; }
  return abort_check();
}

int nfb_selftest_microbench(int mode, int n, int reps, int nwarps, long long* out) {
  using namespace nfb::tc;
  if (!out || n < 16 || n > 256 || n % 16) return fail("microbench: bad arguments");
  if (ensure_abort_flag() || abort_check()) return -1;
  long long* d = nullptr;
  unsigned char* g = nullptr;
  NFB_CUDA(cudaMalloc(&d, 4 * sizeof(long long)));
  NFB_CUDA(cudaMemset(d, 0, 4 * sizeof(long long)));
  NFB_CUDA(cudaMalloc(&g, 8 * 16384));
  NFB_CUDA(cudaMemset(g, 0, 8 * 16384));
  const int smem = ((mode & 255) >= 4 && (mode & 255) <= 6) ? 224 * 1024 : 7 * 16384;
  NFB_CUDA(cudaFuncSetAttribute(tc_microbench_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  // mode bits 9..: grid size minus one (chip-wide contention experiments)
  const int grid = (mode >> 9) + 1;
  mode &= 511;
  tc_microbench_kernel<<<grid, 320, smem>>>(mode, n, reps, nwarps, d, g, smem / 4);
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(g);
  if (e == cudaSuccess) e = cudaMemcpy(out, d, 3 * sizeof(long long), cudaMemcpyDeviceToHost);
  cudaFree(d);
  if (e != cudaSuccess) return fail("microbench failed: %s", cudaGetErrorString(e));
  return abort_check();
}

int nfb_create(const nfb_config* cfg, int max_rays, nfb_handle** out) {
  if (!cfg || !out) return fail("null argument");
  if (max_rays < 1) return fail("max_rays must be >= 1");
  if (cfg->num_coarse_samples < 2) return fail("num_coarse_samples must be >= 2");
  if (cfg->num_fine_samples < 0) return fail("num_fine_samples must be >= 0");
  if (cfg->precision < NFB_PREC_FP32 || cfg->precision > NFB_PREC_FP16X3) return fail("bad precision");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
    return fail("no CUDA device: nerfies_b200 has no CPU path");
  nfb_handle* h = new nfb_handle();
  h->cfg = *cfg;
  h->max_rays = max_rays;
  auto bail = [&](int) { nfb_destroy(h); return -1; };
  if (cudaGetDevice(&h->device) != cudaSuccess) return bail(fail("cudaGetDevice failed"));
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, h->device) != cudaSuccess) return bail(fail("cudaGetDeviceProperties failed"));
  if (prop.major != 10) return bail(fail("device is sm_%d%d; this library is built for sm_100a only", prop.major, prop.minor));
  h->sm_count = prop.multiProcessorCount;
  if (ensure_abort_flag()) return bail(-1);
  if (build_programs(h)) return bail(-1);
  if (build_tables(h)) return bail(-1);
  const nfb_config& c = h->cfg;
  const int nc = c.num_coarse_samples, nfine = nc + c.num_fine_samples;
  auto dmalloc = [&](float** p, long long n) {
    return cudaMalloc(p, (size_t)std::max<long long>(n, 1) * sizeof(float)) == cudaSuccess ? 0
        : fail("cudaMalloc of %lld floats failed", n);
  };
  const long long B = max_rays;
  if (dmalloc(&h->d_packed, h->packed_floats) ||
      dmalloc(&h->d_warp_table, (long long)c.num_warp_embeddings * c.num_warp_features) ||
      dmalloc(&h->d_app_table, (long long)c.num_appearance_embeddings * c.num_appearance_features) ||
      dmalloc(&h->d_cam_table, (long long)c.num_camera_embeddings * c.num_camera_features) ||
      dmalloc(&h->d_cond, B * h->cond_stride) || dmalloc(&h->d_zc, B * nc) ||
      dmalloc(&h->d_zf, B * nfine) || dmalloc(&h->d_wc, B * nc) ||
      dmalloc(&h->d_samples, B * nfine * 4) || dmalloc(&h->d_out_c, B * 6) ||
      dmalloc(&h->d_out_f, B * 6) || dmalloc(&h->d_in, B * 9))
    return bail(-1);
  if (cudaMalloc(&h->d_ids, (size_t)B * 3 * sizeof(unsigned)) != cudaSuccess) return bail(fail("cudaMalloc ids failed"));
  if (cudaMemset(h->d_packed, 0, (size_t)h->packed_floats * sizeof(float)) != cudaSuccess) return bail(fail("cudaMemset failed"));
  if (cudaFuncSetAttribute(nfb::field_simt_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                           nfb::kSimtSmemBytes) != cudaSuccess)
    return bail(fail("cannot reserve %d bytes of shared memory", nfb::kSimtSmemBytes));
  cudaFuncSetAttribute(nfb::composite_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
  cudaFuncSetAttribute(nfb::resample_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024);
#ifdef NFB_WITH_TC
  if (c.precision != NFB_PREC_FP32 && nfb::tc::create_tc(h)) return bail(-1);
  if (c.precision == NFB_PREC_FP16X3 && nfb::tc3::create_x3(h)) return bail(-1);
#endif
  *out = h;
  return 0;
}

void nfb_destroy(nfb_handle* h) {
  if (!h) return;
#ifdef NFB_WITH_TC
  nfb::tc::destroy_tc(h);
#endif
  float* bufs[] = {h->d_packed, h->d_warp_table, h->d_app_table, h->d_cam_table, h->d_zlin,
                   h->d_lower, h->d_upper, h->d_ulin, h->d_window, h->d_cond, h->d_zc, h->d_zf,
                   h->d_wc, h->d_samples, h->d_out_c, h->d_out_f, h->d_in};
  for (float* p : bufs) if (p) cudaFree(p);
  float* tbufs[] = {h->d_tape, h->d_gpacked, h->d_gwarp, h->d_gapp, h->d_gcam, h->d_dcond, h->d_tr_out, h->d_tr_w, h->d_loss,
                    h->d_ttape, reinterpret_cast<float*>(h->d_sel), h->d_time_tape};
  for (float* p : tbufs) if (p) cudaFree(p);
  if (h->d_ids) cudaFree(h->d_ids);
  for (int l = 0; l < 2; ++l)
    for (int i = 0; i < 2; ++i) if (h->ev[l][i]) cudaEventDestroy(h->ev[l][i]);
  if (h->h_in) cudaFreeHost(h->h_in);
  if (h->h_out) cudaFreeHost(h->h_out);
  if (h->h_ids) cudaFreeHost(h->h_ids);
  if (h->ev_order) cudaEventDestroy(h->ev_order);
  delete h;
}

int nfb_param_count(const nfb_handle* h) { return h ? (int)h->specs.size() : fail("null handle"); }

int nfb_param_info(const nfb_handle* h, int index, char* name, int name_capacity,
                   long long* rows, long long* cols) {
  if (!h) return fail("null handle");
  if (index < 0 || index >= (int)h->specs.size()) return fail("parameter index %d out of range", index);
  const ParamSpec& s = h->specs[index];
  if (name && name_capacity > 0) {
    strncpy(name, s.name.c_str(), name_capacity - 1);
    name[name_capacity - 1] = 0;
  }
  if (rows) *rows = s.rows;
  if (cols) *cols = s.cols;
  return 0;
}

int nfb_set_params(nfb_handle* h, const float* const* tensors, const long long* numels,
                   int count, void* stream) {
  if (!h || !tensors || !numels) return fail("null argument");
  if (count != (int)h->specs.size())
    return fail("expected %d parameter tensors, got %d", (int)h->specs.size(), count);
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  for (int i = 0; i < count; ++i) {
    const ParamSpec& p = h->specs[i];
    if (numels[i] != p.rows * p.cols)
      return fail("parameter %d (%s): expected %lld x %lld = %lld elements, got %lld", i,
                  p.name.c_str(), p.rows, p.cols, p.rows * p.cols, numels[i]);
    if (!tensors[i]) return fail("parameter %d (%s) is null", i, p.name.c_str());
    float* base = p.table == 0 ? h->d_packed : p.table == 1 ? h->d_warp_table
                  : p.table == 2 ? h->d_app_table : h->d_cam_table;
    const long long n = p.rows * p.cols;
    if (n == 0) continue;
    pack_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(tensors[i], base + p.dst_off, p.rows,
                                                            p.cols, p.ld, p.c_off);
    if (launch_check(h, "pack_kernel")) return -1;
  }
#ifdef NFB_WITH_TC
  if (h->cfg.precision != NFB_PREC_FP32 && nfb::tc::pack_tc(h, s)) return -1;
#endif
  h->params_set = true;
  return 0;
}

int nfb_coarse_z_vals(nfb_handle* h, int B, const float* t_rand, float* z, void* stream) {
  if (check_call(h, B)) return -1;
  if (B == 0) return 0;
  if (enter_stream(h, (cudaStream_t)stream)) return -1;
  const int nc = h->cfg.num_coarse_samples;
  const long long total = (long long)B * nc;
  nfb::coarse_z_kernel<<<(unsigned)((total + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      h->d_zlin, h->d_lower, h->d_upper, t_rand, z, B, nc);
  return launch_check(h, "coarse_z_kernel");
}

int nfb_sample_pdf(nfb_handle* h, int B, const float* z_coarse, const float* w_coarse,
                   const float* u_rand, float* z_fine, void* stream) {
  if (check_call(h, B)) return -1;
  if (h->cfg.num_fine_samples <= 0) return fail("model has no fine level");
  if (B == 0) return 0;
  if (enter_stream(h, (cudaStream_t)stream)) return -1;
  return run_resample(h, B, z_coarse, w_coarse, u_rand, z_fine, (cudaStream_t)stream);
}

int nfb_render_samples(nfb_handle* h, int level, int B, int S, const float* z_vals,
                       const float* origins, const float* directions, const float* viewdirs,
                       const unsigned* warp_id, const unsigned* app_id, const unsigned* cam_id,
                       float warp_alpha, unsigned flags, float* out, float* weights,
                       float* samples, float* warped_points, void* stream) {
  if (check_call(h, B)) return -1;
  if (level < 0 || level > 1 || (level == 1 && h->cfg.num_fine_samples <= 0)) return fail("bad level %d", level);
  const int smax = h->cfg.num_coarse_samples + h->cfg.num_fine_samples;
  if (S < 1 || (!samples && S > smax)) return fail("num_samples=%d exceeds the workspace (%d)", S, smax);
  if (B == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  if (set_window(h, warp_alpha, s)) return -1;
  if (run_cond(h, B, viewdirs ? viewdirs : directions, warp_id, app_id, cam_id, s,
               (flags & NFB_FLAG_METADATA_ENCODED) != 0)) return -1;
  float* smp = samples ? samples : h->d_samples;
  const bool use_warp = !(flags & NFB_FLAG_NO_WARP);
  if (run_field(h, level, (long long)B * S, S, origins, directions, z_vals, smp, warped_points,
                use_warp, false, s)) return -1;
  if (out) return run_composite(h, B, S, smp, z_vals, directions, out, weights, s);
  return 0;
}

int nfb_render_forward(nfb_handle* h, int B, const float* origins, const float* directions,
                       const float* viewdirs, const unsigned* warp_id, const unsigned* app_id,
                       const unsigned* cam_id, float warp_alpha, const float* t_rand,
                       const float* u_rand, unsigned flags, float* out_coarse, float* out_fine,
                       float* w_coarse, float* w_fine, float* z_fine, void* stream) {
  if (check_call(h, B)) return -1;
  if (B == 0) return 0;
  const nfb_config& c = h->cfg;
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  const int nc = c.num_coarse_samples, nfine = nc + c.num_fine_samples;
  const bool use_warp = !(flags & NFB_FLAG_NO_WARP);
  const bool fine = c.num_fine_samples > 0 && !(flags & NFB_FLAG_COARSE_ONLY);
  if (set_window(h, warp_alpha, s)) return -1;
  if (run_cond(h, B, viewdirs ? viewdirs : directions, warp_id, app_id, cam_id, s,
               (flags & NFB_FLAG_METADATA_ENCODED) != 0)) return -1;
  // coarse level (models.py:332-349)
  if (nfb_coarse_z_vals(h, B, t_rand, h->d_zc, stream)) return -1;
  float* wc = w_coarse ? w_coarse : h->d_wc;
  float* oc = out_coarse ? out_coarse : h->d_out_c;
  if (can_fuse_composite(h, nc)) {
    // field + volumetric rendering in one kernel: 24 B per ray (+ the coarse weights) leave the SM
    if (run_field(h, 0, (long long)B * nc, nc, origins, directions, h->d_zc, nullptr, nullptr,
                  use_warp, false, s, oc, wc)) return -1;
  } else {
    if (run_field(h, 0, (long long)B * nc, nc, origins, directions, h->d_zc, h->d_samples, nullptr,
                  use_warp, false, s)) return -1;
    if (run_composite(h, B, nc, h->d_samples, h->d_zc, directions, oc, wc, s)) return -1;
  }
  if (!fine) return 0;
  // hierarchical resampling + fine level (models.py:352-370)
  float* zf = z_fine ? z_fine : h->d_zf;
  if (run_resample(h, B, h->d_zc, wc, u_rand, zf, s)) return -1;
  float* of = out_fine ? out_fine : h->d_out_f;
  if (can_fuse_composite(h, nfine))
    return run_field(h, 1, (long long)B * nfine, nfine, origins, directions, zf, nullptr, nullptr,
                     use_warp, false, s, of, w_fine);
  if (run_field(h, 1, (long long)B * nfine, nfine, origins, directions, zf, h->d_samples, nullptr,
                use_warp, false, s)) return -1;
  return run_composite(h, B, nfine, h->d_samples, zf, directions, of, w_fine, s);
}

int nfb_render_forward_host(nfb_handle* h, int B, const float* origins, const float* directions,
                            const float* viewdirs, const unsigned* warp_id,
                            const unsigned* app_id, const unsigned* cam_id, float warp_alpha,
                            unsigned flags, float* out_coarse, float* out_fine, void* stream) {
  if (check_call(h, B)) return -1;
  if (flags & NFB_FLAG_METADATA_ENCODED)
    return fail("NFB_FLAG_METADATA_ENCODED is only supported by the device entry points");
  if (B == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  const size_t mr = h->max_rays;
  // (each buffer on its own: a failed allocation leaves the others usable for the retry)
  if (!h->h_in) NFB_CUDA(cudaMallocHost(&h->h_in, mr * 9 * sizeof(float)));
  if (!h->h_out) NFB_CUDA(cudaMallocHost(&h->h_out, mr * 12 * sizeof(float)));
  if (!h->h_ids) NFB_CUDA(cudaMallocHost(&h->h_ids, mr * 3 * sizeof(unsigned)));
  const size_t n3 = (size_t)B * 3;
  memcpy(h->h_in, origins, n3 * sizeof(float));
  memcpy(h->h_in + mr * 3, directions, n3 * sizeof(float));
  if (viewdirs) memcpy(h->h_in + mr * 6, viewdirs, n3 * sizeof(float));
  const unsigned* ids[3] = {warp_id, app_id, cam_id};
  for (int i = 0; i < 3; ++i)
    if (ids[i]) memcpy(h->h_ids + mr * i, ids[i], (size_t)B * sizeof(unsigned));
  NFB_CUDA(cudaMemcpyAsync(h->d_in, h->h_in, n3 * sizeof(float), cudaMemcpyHostToDevice, s));
  NFB_CUDA(cudaMemcpyAsync(h->d_in + mr * 3, h->h_in + mr * 3, n3 * sizeof(float), cudaMemcpyHostToDevice, s));
  if (viewdirs)
    NFB_CUDA(cudaMemcpyAsync(h->d_in + mr * 6, h->h_in + mr * 6, n3 * sizeof(float), cudaMemcpyHostToDevice, s));
  for (int i = 0; i < 3; ++i)
    if (ids[i])
      NFB_CUDA(cudaMemcpyAsync(h->d_ids + mr * i, h->h_ids + mr * i, (size_t)B * sizeof(unsigned),
                               cudaMemcpyHostToDevice, s));
  if (nfb_render_forward(h, B, h->d_in, h->d_in + mr * 3, viewdirs ? h->d_in + mr * 6 : nullptr,
                         warp_id ? h->d_ids : nullptr, app_id ? h->d_ids + mr : nullptr,
                         cam_id ? h->d_ids + 2 * mr : nullptr, warp_alpha, nullptr, nullptr, flags,
                         h->d_out_c, h->d_out_f, nullptr, nullptr, nullptr, stream))
    return -1;
  const bool fine = h->cfg.num_fine_samples > 0 && !(flags & NFB_FLAG_COARSE_ONLY);
  if (out_coarse)
    NFB_CUDA(cudaMemcpyAsync(h->h_out, h->d_out_c, (size_t)B * 6 * sizeof(float), cudaMemcpyDeviceToHost, s));
  if (out_fine && fine)
    NFB_CUDA(cudaMemcpyAsync(h->h_out + mr * 6, h->d_out_f, (size_t)B * 6 * sizeof(float), cudaMemcpyDeviceToHost, s));
  NFB_CUDA(cudaStreamSynchronize(s));
  if (abort_check()) return -1;
  if (out_coarse) memcpy(out_coarse, h->h_out, (size_t)B * 6 * sizeof(float));
  if (out_fine && fine) memcpy(out_fine, h->h_out + mr * 6, (size_t)B * 6 * sizeof(float));
  return 0;
}

int nfb_warp_forward(nfb_handle* h, int P, const float* points, const unsigned* warp_id,
                     float warp_alpha, unsigned flags, float* warped, void* stream) {
  if (check_call(h, P)) return -1;
  if (h->cfg.warp_field_type == NFB_WARP_NONE) return fail("model has no warp field");
  if (P == 0) return 0;
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  if (set_window(h, warp_alpha, s)) return -1;
  // Only the GLO block of the condition vector is read in warp-only mode; the
  // view-direction block is computed from `points` and ignored.
  if (run_cond(h, P, points, warp_id, nullptr, nullptr, s, (flags & NFB_FLAG_METADATA_ENCODED) != 0)) return -1;
  // Free points: rows = points, z = 0 (x = p + 0 * p = p exactly for finite p).
  return run_field(h, 0, P, 1, points, points, nullptr, nullptr, warped, true, true, s);
}

}  // extern "C"

#include "train_api.cuh"
