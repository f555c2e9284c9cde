// Host side of the training tier: tape layout, the forward / backward launch
// sequence of one level, nfb_train_value_and_grad and nfb_adam_step
// (see train.cuh; included by nfb_api.cu after its helpers).
#pragma once
#include "train.cuh"
#include "train_reg.cuh"

namespace {

using nfb::Net;
using nfb::Step;

// Step s reads the output of step producer[s] (or nothing when k_x == 0).
void net_producers(const Net& net, int* producer) {
  int writer[4] = {-1, -1, -1, -1};
  for (int s = 0; s < net.n_steps; ++s) {
    producer[s] = net.steps[s].k_x > 0 ? writer[net.steps[s].src] : -1;
    writer[net.steps[s].dst] = s;
  }
}

struct TapeLayout {
  long long rows = 0;
  // float offsets into the arena
  long long pts = 0, warped = 0, in_w = 0, in_n = 0, samples = 0, dwarped = 0, d_in_w = 0, d_in_n = 0;
  long long out_w[nfb::kMaxSteps], out_n[nfb::kMaxSteps], d_out_w[nfb::kMaxSteps], d_out_n[nfb::kMaxSteps];
  long long grad_begin = 0, grad_end = 0, total = 0;
  int ld_w = 0, ld_n = 0;
};

TapeLayout tape_layout(const nfb::FieldProgram& p, long long rows) {
  TapeLayout t;
  t.rows = rows;
  long long off = 0;
  auto take = [&](long long n) { long long o = off; off += (n + 63) / 64 * 64; return o; };
  t.ld_w = pad32(p.Dw);
  t.ld_n = pad32(p.Dp + p.tc + p.ac + p.rc);
  t.pts = take(rows * 3); t.warped = take(rows * 3);
  t.in_w = take(rows * t.ld_w); t.in_n = take(rows * t.ld_n);
  t.samples = take(rows * 4);
  for (int s = 0; s < p.warp.n_steps; ++s) t.out_w[s] = take(rows * p.warp.steps[s].npad);
  for (int s = 0; s < p.nerf.n_steps; ++s) t.out_n[s] = take(rows * p.nerf.steps[s].npad);
  t.grad_begin = off;
  t.dwarped = take(rows * 3);
  t.d_in_w = take(rows * t.ld_w); t.d_in_n = take(rows * t.ld_n);
  for (int s = 0; s < p.warp.n_steps; ++s) t.d_out_w[s] = take(rows * p.warp.steps[s].npad);
  for (int s = 0; s < p.nerf.n_steps; ++s) t.d_out_n[s] = take(rows * p.nerf.steps[s].npad);
  t.grad_end = off;
  t.total = off;
  return t;
}

// Rows per split of a weight-gradient GEMM (reduction over the rows of the batch; the partial tiles are
// atomicAdd-ed).  The output is tiny (<= 3 x 2 tiles of 128 x 128), so the split count sets the parallelism:
// aim at ~4 CTAs per resident slot (2 per SM) whatever the layer's width; a fixed 2048 rows left a 128-wide
// layer of a 131,072-row chunk with 64 CTAs for 148 SMs, 8192 rows measured 3x slower.
inline long long dw_split(const nfb_handle* h, long long M, int N, long long K) {
  const long long tiles = ((M + nfb::train::kT2 - 1) / nfb::train::kT2) * ((N + nfb::train::kT2 - 1) / nfb::train::kT2);
  const long long want = std::max<long long>(1, (8LL * h->sm_count) / tiles);   // splits
  long long per = (K + want - 1) / want;
  per = (per + 7) / 8 * 8;
  return std::min<long long>(4096, std::max<long long>(256, per));
}
// kAKFast / kBNFast: see sgemm128_kernel (which functor index is contiguous in memory).
template <bool kAKFast = true, bool kBNFast = true, class FA, class FB, class FC>
int launch_gemm(nfb_handle* h, long long M, int N, long long K, FA fa, FB fb, FC fc, long long k_split,
                cudaStream_t s, const char* what) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  const long long per = k_split > 0 ? k_split : K;
#ifdef NFB_TRAIN_SGEMM64
  dim3 grid((unsigned)((M + nfb::train::kTile - 1) / nfb::train::kTile),
            (unsigned)((N + nfb::train::kTile - 1) / nfb::train::kTile), (unsigned)((K + per - 1) / per));
  nfb::train::sgemm_kernel<<<grid, 256, 0, s>>>(nfb::train::GemmShape{M, N, K}, fa, fb, fc, per);
#else
  dim3 grid((unsigned)((M + nfb::train::kT2 - 1) / nfb::train::kT2),
            (unsigned)((N + nfb::train::kT2 - 1) / nfb::train::kT2), (unsigned)((K + per - 1) / per));
  nfb::train::sgemm128_kernel<kAKFast, kBNFast><<<grid, 256, 0, s>>>(nfb::train::GemmShape{M, N, K}, fa, fb, fc, per);
#endif
  return launch_check(h, what);
}

int net_forward(nfb_handle* h, const Net& net, const float* in, int ld_in, const long long* out_off,
                float* arena, long long rows, cudaStream_t s) {
  int producer[nfb::kMaxSteps];
  net_producers(net, producer);
  for (int i = 0; i < net.n_steps; ++i) {
    const Step& st = net.steps[i];
    const float* x = producer[i] >= 0 ? arena + out_off[producer[i]] : in;
    const int ldx = producer[i] >= 0 ? net.steps[producer[i]].npad : ld_in;
    nfb::train::ConcatA a{x, ldx, st.k_x, in + st.in_off, ld_in};
    nfb::train::WeightB b{h->d_packed + st.w_off, st.npad};
    nfb::train::StoreBiasAct c{arena + out_off[i], st.npad, h->d_packed + st.b_off, st.act};
    if (launch_gemm(h, rows, st.n, st.k_x + st.k_in, a, b, c, 0, s, "sgemm (forward)")) return -1;
  }
  return 0;
}

int net_backward(nfb_handle* h, const Net& net, const float* in, float* d_in, int ld_in,
                 const long long* out_off, const long long* d_out_off, float* arena, long long rows,
                 cudaStream_t s) {
  int producer[nfb::kMaxSteps];
  net_producers(net, producer);
  for (int i = net.n_steps - 1; i >= 0; --i) {
    const Step& st = net.steps[i];
    const int K = st.k_x + st.k_in;
    nfb::train::DZ dz{arena + d_out_off[i], arena + out_off[i], st.npad, st.act};
    const float* x = producer[i] >= 0 ? arena + out_off[producer[i]] : in;
    const int ldx = producer[i] >= 0 ? net.steps[producer[i]].npad : ld_in;
    nfb::train::ConcatA a{x, ldx, st.k_x, in + st.in_off, ld_in};
    // dW += [X | IN]^T dZ   (reduction over the rows, split)
    if (launch_gemm<false, true>(h, K, st.n, rows, nfb::train::ConcatAT{a}, nfb::train::DZB{dz},
                                 nfb::train::AtomicAdd{h->d_gpacked + st.w_off, st.npad}, dw_split(h, K, st.n, rows), s, "sgemm (dW)")) return -1;
    // db += colsum(dZ)
    {
      dim3 grid((unsigned)((st.n + 31) / 32), (unsigned)std::min<long long>((rows + 255) / 256, 128));
      nfb::train::colsum_kernel<<<grid, 256, 0, s>>>(dz, rows, st.n, h->d_gpacked + st.b_off);
      if (launch_check(h, "colsum_kernel")) return -1;
    }
    // dX, dIN += dZ W^T
    float* dx = producer[i] >= 0 ? arena + d_out_off[producer[i]] : d_in;
    nfb::train::AccumSplit acc{dx, ldx, st.k_x, d_in + st.in_off, ld_in};
    if (launch_gemm<true, false>(h, rows, K, st.n, dz, nfb::train::WeightBT{h->d_packed + st.w_off, st.npad}, acc, 0, s,
                                 "sgemm (dX)")) return -1;
  }
  return 0;
}

// ---- tangent tape (train_reg.cuh): three rows per selected point ----
struct TTapeLayout {
  long long trows = 0;
  long long in_t = 0, d_in_t = 0, total = 0;
  long long out_t[nfb::kMaxSteps], d_out_t[nfb::kMaxSteps];
};
TTapeLayout ttape_layout(const nfb::FieldProgram& p, long long sel_rows) {
  TTapeLayout t;
  t.trows = sel_rows * 3;
  long long off = 0;
  auto take = [&](long long n) { long long o = off; off += (n + 63) / 64 * 64; return o; };
  const int ld_w = pad32(p.Dw);
  t.in_t = take(t.trows * ld_w); t.d_in_t = take(t.trows * ld_w);
  for (int s = 0; s < p.warp.n_steps; ++s) { t.out_t[s] = take(t.trows * p.warp.steps[s].npad); t.d_out_t[s] = take(t.trows * p.warp.steps[s].npad); }
  t.total = off;
  return t;
}
int ensure_ttape(nfb_handle* h, long long floats, long long sel_rows) {
  if (h->ttape_floats < floats) {
    if (h->d_ttape) cudaFree(h->d_ttape);
    h->d_ttape = nullptr; h->ttape_floats = 0;
    if (cudaMalloc(&h->d_ttape, (size_t)floats * sizeof(float)) != cudaSuccess)
      return fail("training: cannot allocate a %.2f GB tangent tape", floats * 4e-9);
    h->ttape_floats = floats;
  }
  if (h->sel_cap < sel_rows) {
    if (h->d_sel) cudaFree(h->d_sel);
    h->d_sel = nullptr; h->sel_cap = 0;
    if (cudaMalloc(&h->d_sel, (size_t)sel_rows * sizeof(int)) != cudaSuccess) return fail("training: cudaMalloc failed");
    h->sel_cap = sel_rows;
  }
  return 0;
}

// Tangent rows through the warp MLP: T_out = act'(Y_primal) * ([T_x | T_in] W).
int tnet_forward(nfb_handle* h, const Net& net, const float* tin, int ld_in, const long long* out_t,
                 const long long* out_primal, const float* arena, float* tarena, const int* sel, long long trows,
                 cudaStream_t s) {
  int producer[nfb::kMaxSteps];
  net_producers(net, producer);
  for (int i = 0; i < net.n_steps; ++i) {
    const Step& st = net.steps[i];
    const float* x = producer[i] >= 0 ? tarena + out_t[producer[i]] : tin;
    const int ldx = producer[i] >= 0 ? net.steps[producer[i]].npad : ld_in;
    nfb::train::ConcatA a{x, ldx, st.k_x, tin + st.in_off, ld_in};
    nfb::train::WeightB b{h->d_packed + st.w_off, st.npad};
    nfb::train::StoreMasked c{tarena + out_t[i], st.npad, arena + out_primal[i], sel, st.act};
    if (launch_gemm(h, trows, st.n, st.k_x + st.k_in, a, b, c, 0, s, "sgemm (tangent forward)")) return -1;
  }
  return 0;
}
// ... and backwards: weight gradients only (no bias; the masks are piecewise constant).
int tnet_backward(nfb_handle* h, const Net& net, const float* tin, float* d_tin, int ld_in, const long long* out_t,
                  const long long* d_out_t, const long long* out_primal, const float* arena, float* tarena,
                  const int* sel, long long trows, cudaStream_t s) {
  int producer[nfb::kMaxSteps];
  net_producers(net, producer);
  for (int i = net.n_steps - 1; i >= 0; --i) {
    const Step& st = net.steps[i];
    const int K = st.k_x + st.k_in;
    nfb::train::DZT dz{tarena + d_out_t[i], arena + out_primal[i], sel, st.npad, st.act};
    const float* x = producer[i] >= 0 ? tarena + out_t[producer[i]] : tin;
    const int ldx = producer[i] >= 0 ? net.steps[producer[i]].npad : ld_in;
    nfb::train::ConcatA a{x, ldx, st.k_x, tin + st.in_off, ld_in};
    if (launch_gemm<false, true>(h, K, st.n, trows, nfb::train::ConcatAT{a}, nfb::train::DZTB{dz},
                                 nfb::train::AtomicAdd{h->d_gpacked + st.w_off, st.npad}, dw_split(h, K, st.n, trows), s, "sgemm (tangent dW)")) return -1;
    if (i == 0 && st.k_x == 0) break;             // nothing upstream of the encoded input carries a parameter
    float* dx = producer[i] >= 0 ? tarena + d_out_t[producer[i]] : d_tin;
    nfb::train::AccumSplit acc{dx, ldx, st.k_x, d_tin + st.in_off, ld_in};
    if (launch_gemm<true, false>(h, trows, K, st.n, dz, nfb::train::WeightBT{h->d_packed + st.w_off, st.npad}, acc, 0, s,
                                 "sgemm (tangent dX)")) return -1;
  }
  return 0;
}

// Regularisers of one training step (training.py:138-147, 176-212, 246-257).
struct RegCfg {
  bool elastic = false; int reduce = 0, type = 0; float elastic_weight = 0.f;
  bool warp_reg = false; float warp_reg_weight = 0.f, warp_reg_alpha = -2.f, warp_reg_scale = 0.001f;
  int batch_rays = 1;             // rays of the whole local batch (the means are over it)
  float* stats = nullptr;         // device: nfb_train_value_and_grad_reg's loss_out layout
};

// Jacobian (+ elastic loss and its adjoint when `with_grad`) at `sel_rows` tape rows of the warp tape in `A`.
int warp_jacobian_on_tape(nfb_handle* h, const nfb::FieldProgram& p, const TapeLayout& t, float* A, const int* sel,
                          long long sel_rows, const float* row_w, const RegCfg* reg, bool with_grad, float* jac_out,
                          cudaStream_t s) {
  using namespace nfb::train;
  for (int i = 0; i < p.warp.n_steps - 1; ++i)
    if (p.warp.steps[i].act != nfb::kRelu && p.warp.steps[i].act != nfb::kNone)
      return fail("warp Jacobian: the warp MLP must use relu (piecewise-linear) activations");
  const TTapeLayout tt = ttape_layout(p, sel_rows);
  if (ensure_ttape(h, tt.total, 1)) return -1;
  float* T = h->d_ttape;
  if (with_grad) NFB_CUDA(cudaMemsetAsync(T + tt.d_in_t, 0, (size_t)(tt.total - tt.d_in_t) * sizeof(float), s));
  const unsigned tblocks = (unsigned)((tt.trows + 127) / 128);
  EncodeTangentArgs e{A + t.pts, sel, h->d_window, T + tt.in_t, p.Fw, t.ld_w, sel_rows};
  encode_tangent_kernel<<<tblocks, 128, 0, s>>>(e);
  if (launch_check(h, "encode_tangent_kernel")) return -1;
  if (tnet_forward(h, p.warp, T + tt.in_t, t.ld_w, tt.out_t, t.out_w, A, T, sel, tt.trows, s)) return -1;
  const int hs = p.warp.n_steps - 1;
  JacArgs j{};
  j.head = A + t.out_w[hs]; j.ld = p.warp.steps[hs].npad; j.thead = T + tt.out_t[hs]; j.pts = A + t.pts;
  j.sel = sel; j.row_w = row_w; j.jac_out = jac_out; j.R = sel_rows;
  j.warp_type = p.warp_type; j.pivot = p.warp_pivot; j.trans = p.warp_trans;
  j.with_loss = reg != nullptr; j.loss_type = reg ? reg->type : 0;
  j.stats = reg ? reg->stats + 2 : nullptr;
  if (with_grad) {
    j.d_head = A + t.d_out_w[hs]; j.d_thead = T + tt.d_out_t[hs];
    j.grad_scale = reg->elastic_weight / (float)reg->batch_rays;
  }
  jac_elastic_kernel<<<(unsigned)((sel_rows + 63) / 64), 64, 0, s>>>(j);
  if (launch_check(h, "jac_elastic_kernel")) return -1;
  if (with_grad &&
      tnet_backward(h, p.warp, T + tt.in_t, T + tt.d_in_t, t.ld_w, tt.out_t, tt.d_out_t, t.out_w, A, T, sel,
                    tt.trows, s))
    return -1;
  return 0;
}

// forward + loss + backward of one level for `R` rays (rows = R * S) on the tape.
int train_level(nfb_handle* h, int level, int R, int S, const float* z, const float* origins,
                const float* directions, const float* target, float scale, bool use_warp,
                float* out6, float* weights, float* loss, cudaStream_t s, const RegCfg* reg = nullptr) {
  using namespace nfb::train;
  const nfb::FieldProgram& p = h->prog[level];
  const long long rows = (long long)R * S;
  const TapeLayout t = tape_layout(p, rows);
  float* A = h->d_tape;
  const bool warp = use_warp && p.warp_type != 0;
  const unsigned blocks = (unsigned)((rows + 127) / 128);
  // ---- forward ----
  if (warp) {
    EncodeArgs e{};
    e.origins = origins; e.directions = directions; e.z = z; e.cond = h->d_cond; e.window = h->d_window;
    e.pts_out = A + t.pts; e.in = A + t.in_w; e.F = p.Fw; e.ld = t.ld_w; e.S = S;
    e.cond_stride = h->cond_stride; e.cond_off = 0; e.n_cond = p.G; e.rows = rows;
    encode_kernel<<<blocks, 128, 0, s>>>(e);
    if (launch_check(h, "encode_kernel")) return -1;
    if (net_forward(h, p.warp, A + t.in_w, t.ld_w, t.out_w, A, rows, s)) return -1;
    const int hs = p.warp.n_steps - 1;
    WarpTailArgs w{A + t.out_w[hs], p.warp.steps[hs].npad, A + t.pts, A + t.warped, p.warp_type, p.warp_pivot,
                   p.warp_trans, rows};
    warp_tail_kernel<<<blocks, 128, 0, s>>>(w);
    if (launch_check(h, "warp_tail_kernel")) return -1;
  }
  {
    EncodeArgs e{};
    e.origins = origins; e.directions = directions; e.z = z; e.cond = h->d_cond; e.window = nullptr;
    e.pts_in = warp ? A + t.warped : nullptr; e.pts_out = warp ? nullptr : A + t.warped;
    e.in = A + t.in_n; e.F = p.Fp; e.ld = t.ld_n; e.S = S;
    e.cond_stride = h->cond_stride; e.cond_off = p.G; e.n_cond = p.tc + p.ac + p.rc; e.rows = rows;
    encode_kernel<<<blocks, 128, 0, s>>>(e);
    if (launch_check(h, "encode_kernel")) return -1;
  }
  if (net_forward(h, p.nerf, A + t.in_n, t.ld_n, t.out_n, A, rows, s)) return -1;
  // which steps hold the raw alpha / rgb (the last writers of the two output slots)
  int alpha_step = -1, rgb_step = -1;
  for (int i = 0; i < p.nerf.n_steps; ++i) {
    if (p.nerf.steps[i].dst == p.alpha_slot) alpha_step = i;
    if (p.nerf.steps[i].dst == p.rgb_slot) rgb_step = i;
  }
  if (alpha_step < 0 || rgb_step < 0) return fail("training: no alpha / rgb head in the program");
  const int ld_a = p.nerf.steps[alpha_step].npad, ld_rgb = p.nerf.steps[rgb_step].npad;
  raw_to_samples_kernel<<<blocks, 128, 0, s>>>(A + t.out_n[rgb_step], ld_rgb, A + t.out_n[alpha_step], ld_a,
                                               p.sigma_act, reinterpret_cast<float4*>(A + t.samples), rows);
  if (launch_check(h, "raw_to_samples_kernel")) return -1;
  if (run_composite(h, R, S, A + t.samples, z, directions, out6, weights, s)) return -1;
  // ---- loss + backward ----
  NFB_CUDA(cudaMemsetAsync(A + t.grad_begin, 0, (size_t)(t.grad_end - t.grad_begin) * sizeof(float), s));
  {
    CompositeBwdArgs c{};
    c.samples = reinterpret_cast<const float4*>(A + t.samples); c.z = z; c.directions = directions;
    c.out = out6; c.target = target;
    c.rgb_raw = A + t.out_n[rgb_step]; c.ld_rgb = ld_rgb; c.alpha_raw = A + t.out_n[alpha_step]; c.ld_a = ld_a;
    c.d_rgb_raw = A + t.d_out_n[rgb_step]; c.d_alpha_raw = A + t.d_out_n[alpha_step];
    c.loss = loss; c.scale = scale; c.num_rays = R; c.S = S;
    c.white_bg = h->cfg.use_white_background; c.sample_at_infinity = h->cfg.use_sample_at_infinity;
    c.sigma_act = p.sigma_act;
    const int nblk = (R + nfb::kRaysPerBlock - 1) / nfb::kRaysPerBlock;
    const size_t smem = (size_t)nfb::kRaysPerBlock * 4 * S * sizeof(float);
    composite_bwd_kernel<<<nblk, 32 * nfb::kRaysPerBlock, smem, s>>>(c);
    if (launch_check(h, "composite_bwd_kernel")) return -1;
  }
  const bool want_sel = reg && warp && ((reg->elastic && level == 0 && reg->reduce == 0) || reg->warp_reg);
  if (want_sel) {
    if (ensure_ttape(h, 0, R)) return -1;
    depth_index_kernel<<<(unsigned)((R + 7) / 8), 256, 0, s>>>(weights, R, S, h->d_sel);
    if (launch_check(h, "depth_index_kernel")) return -1;
  }
  if (reg && reg->elastic && level == 0 && warp) {
    // training.py:176-193 (the coarse level only: training.py:242-244)
    const bool median = reg->reduce == 0;
    if (warp_jacobian_on_tape(h, p, t, A, median ? h->d_sel : nullptr, median ? R : rows, median ? nullptr : weights,
                              reg, true, nullptr, s))
      return -1;
  }
  if (net_backward(h, p.nerf, A + t.in_n, A + t.d_in_n, t.ld_n, t.out_n, t.d_out_n, A, rows, s)) return -1;
  {
    EncodeBwdArgs e{};
    e.pts = A + t.warped; e.window = nullptr; e.din = A + t.d_in_n; e.F = p.Fp; e.ld = t.ld_n; e.S = S;
    e.cond_stride = h->cond_stride; e.cond_off = p.G; e.n_cond = p.tc + p.ac + p.rc;
    e.dpts = warp ? A + t.dwarped : nullptr; e.dcond = h->d_dcond; e.rows = rows;
    encode_bwd_kernel<<<blocks, 128, 0, s>>>(e);
    if (launch_check(h, "encode_bwd_kernel")) return -1;
  }
  if (warp && reg && reg->warp_reg) {
    // training.py:194-207: robust loss of |points - warped_points|^2 at the median-depth sample
    WarpMagArgs wm{A + t.pts, A + t.warped, h->d_sel, A + t.dwarped, reg->stats + (level == 0 ? 7 : 9),
                   reg->warp_reg_alpha, reg->warp_reg_scale, reg->warp_reg_weight / (float)reg->batch_rays, R};
    warp_mag_loss_kernel<<<(unsigned)((R + 127) / 128), 128, 0, s>>>(wm);
    if (launch_check(h, "warp_mag_loss_kernel")) return -1;
  }
  if (warp) {
    const int hs = p.warp.n_steps - 1;
    WarpTailBwdArgs w{A + t.out_w[hs], p.warp.steps[hs].npad, A + t.pts, A + t.dwarped, A + t.d_out_w[hs],
                      p.warp_type, p.warp_pivot, p.warp_trans, rows};
    warp_tail_bwd_kernel<<<blocks, 128, 0, s>>>(w);
    if (launch_check(h, "warp_tail_bwd_kernel")) return -1;
    if (net_backward(h, p.warp, A + t.in_w, A + t.d_in_w, t.ld_w, t.out_w, t.d_out_w, A, rows, s)) return -1;
    EncodeBwdArgs e{};
    e.pts = A + t.pts; e.window = h->d_window; e.din = A + t.d_in_w; e.F = p.Fw; e.ld = t.ld_w; e.S = S;
    e.cond_stride = h->cond_stride; e.cond_off = 0; e.n_cond = p.G; e.dpts = nullptr; e.dcond = h->d_dcond;
    e.rows = rows;
    encode_bwd_kernel<<<blocks, 128, 0, s>>>(e);
    if (launch_check(h, "encode_bwd_kernel")) return -1;
  }
  return 0;
}

int train_prepare(nfb_handle* h, int chunk_rays) {
  const nfb_config& c = h->cfg;
  const int smax = c.num_coarse_samples + c.num_fine_samples;
  long long need = 0;
  for (int lv = 0; lv < 2; ++lv) need = std::max(need, tape_layout(h->prog[lv], (long long)chunk_rays * smax).total);
  if (h->tape_floats < need) {
    if (h->d_tape) cudaFree(h->d_tape);
    h->d_tape = nullptr; h->tape_floats = 0;
    if (cudaMalloc(&h->d_tape, (size_t)need * sizeof(float)) != cudaSuccess)
      return fail("training: cannot allocate a %.1f GB tape for %d rays per chunk", need * 4e-9, chunk_rays);
    NFB_CUDA(cudaMemset(h->d_tape, 0, (size_t)need * sizeof(float)));
    h->tape_floats = need;
  }
  cudaFuncSetAttribute(nfb::train::composite_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  if (!h->d_gpacked) {
    auto dm = [&](float** p, long long n) {
      return cudaMalloc(p, (size_t)std::max<long long>(n, 1) * sizeof(float)) == cudaSuccess ? 0
          : fail("training: cudaMalloc of %lld floats failed", n);
    };
    if (dm(&h->d_gpacked, h->packed_floats) ||
        dm(&h->d_gwarp, (long long)c.num_warp_embeddings * c.num_warp_features) ||
        dm(&h->d_gapp, (long long)c.num_appearance_embeddings * c.num_appearance_features) ||
        dm(&h->d_gcam, (long long)c.num_camera_embeddings * c.num_camera_features) ||
        dm(&h->d_dcond, (long long)h->max_rays * h->cond_stride) || dm(&h->d_tr_out, (long long)h->max_rays * 12) ||
        dm(&h->d_tr_w, (long long)h->max_rays * smax) || dm(&h->d_loss, 16))
      return -1;
  }
  return 0;
}

// Tape large enough for `rows` rows of either level (free points: one row per point).
int train_prepare_rows(nfb_handle* h, long long rows) {
  const int smax = h->cfg.num_coarse_samples + h->cfg.num_fine_samples;
  return train_prepare(h, (int)std::max<long long>(1, (rows + smax - 1) / smax));
}

// The GLO side of the warp block of the condition gradient (CondBwdArgs::warp_glo / warp_scale).
void set_warp_glo(const nfb_handle* h, nfb::train::CondBwdArgs& a) {
  const int enc = h->cfg.warp_metadata_encoder;
  a.warp_glo = enc != NFB_WARP_ENC_TIME;
  a.warp_scale = enc == NFB_WARP_ENC_BLEND ? 1.f - h->time_alpha : 1.f;
}

// TimeEncoder backward (modules.py:297-322) for `rows` condition vectors whose warp-block gradient
// d_dcond[:, 0:G] is complete: the encoder's input rows onto its own tape, its forward recomputed
// layer-wise, then dW / db accumulated into d_gpacked at the encoder's offsets.  The recomputed
// activations can differ from time_embed_kernel's in round-off only, so a ReLU mask can differ only
// on a pre-activation within round-off of zero.  `warp_id` / `time_from_ids` as for run_cond.
int time_encoder_backward(nfb_handle* h, int rows, const unsigned* warp_id, bool time_from_ids, cudaStream_t s) {
  using namespace nfb::train;
  const nfb_config& c = h->cfg;
  const int enc = c.warp_metadata_encoder;
  if (c.warp_field_type == NFB_WARP_NONE || enc == NFB_WARP_ENC_GLO || rows == 0) return 0;
  const Net& net = h->time_net;
  const int F = c.time_encoder_num_freqs, ld_in = 1 + 2 * F, last = net.n_steps - 1;
  // input rows, every layer's output, then the gradient region: every layer's dY and the input's
  // gradient (written by the first layer's dX GEMM, not needed)
  long long off = 0, out[nfb::kMaxSteps], d_out[nfb::kMaxSteps];
  auto take = [&](long long n) { long long o = off; off += (n + 63) / 64 * 64; return o; };
  const long long in = take((long long)rows * ld_in);
  for (int i = 0; i < net.n_steps; ++i) out[i] = take((long long)rows * net.steps[i].npad);
  const long long grad_begin = off;
  for (int i = 0; i < net.n_steps; ++i) d_out[i] = take((long long)rows * net.steps[i].npad);
  const long long d_in = take((long long)rows * ld_in);
  if (h->time_tape_floats < off) {
    if (h->d_time_tape) cudaFree(h->d_time_tape);
    h->d_time_tape = nullptr; h->time_tape_floats = 0;
    if (cudaMalloc(&h->d_time_tape, (size_t)off * sizeof(float)) != cudaSuccess)
      return fail("training: cannot allocate a %.2f GB TimeEncoder tape", off * 4e-9);
    h->time_tape_floats = off;
  }
  float* T = h->d_time_tape;
  NFB_CUDA(cudaMemsetAsync(T + grad_begin, 0, (size_t)(off - grad_begin) * sizeof(float), s));
  TimeTapeArgs a{};
  if (enc == NFB_WARP_ENC_TIME && !time_from_ids) a.time_f = reinterpret_cast<const float*>(warp_id);
  else a.time_id = warp_id;
  a.F = F;
  time_window(h, a.window);
  a.dcond = h->d_dcond; a.cond_stride = h->cond_stride; a.G = h->prog[0].G;
  a.seed_scale = enc == NFB_WARP_ENC_BLEND ? h->time_alpha : 1.f;      // warping.py:132-133
  a.in = T + in; a.ld_in = ld_in; a.seed = T + d_out[last]; a.ld_seed = net.steps[last].npad; a.rows = rows;
  time_tape_kernel<<<(unsigned)((rows + 127) / 128), 128, 0, s>>>(a);
  if (launch_check(h, "time_tape_kernel")) return -1;
  if (net_forward(h, net, T + in, ld_in, out, T, rows, s)) return -1;
  return net_backward(h, net, T + in, T + d_in, ld_in, out, d_out, T, rows, s);
}

// warp_field.apply on `n` free points (+ optional noise) on the tape of level 0: condition
// vectors per point, encoded inputs, warp MLP, tail.  The points land in tape.pts, the warped
// points in tape.warped.  `time_from_ids` as for run_cond.
int warp_points_forward(nfb_handle* h, int n, const float* points, const float* noise, const unsigned* warp_id,
                        bool time_from_ids, cudaStream_t s) {
  using namespace nfb::train;
  const nfb::FieldProgram& p = h->prog[0];
  const TapeLayout t = tape_layout(p, n);
  float* A = h->d_tape;
  const unsigned blocks = (unsigned)((n + 127) / 128);
  add_noise_kernel<<<(unsigned)(((long long)n * 3 + 255) / 256), 256, 0, s>>>(points, noise, A + t.warped, (long long)n * 3);
  if (launch_check(h, "add_noise_kernel")) return -1;
  // the "view direction" columns are unused here
  if (run_cond(h, n, A + t.warped, warp_id, nullptr, nullptr, s, false, time_from_ids)) return -1;
  EncodeArgs e{};
  e.pts_in = A + t.warped; e.pts_out = A + t.pts; e.cond = h->d_cond; e.window = h->d_window;
  e.in = A + t.in_w; e.F = p.Fw; e.ld = t.ld_w; e.S = 1;
  e.cond_stride = h->cond_stride; e.cond_off = 0; e.n_cond = p.G; e.rows = n;
  encode_kernel<<<blocks, 128, 0, s>>>(e);
  if (launch_check(h, "encode_kernel")) return -1;
  if (net_forward(h, p.warp, A + t.in_w, t.ld_w, t.out_w, A, n, s)) return -1;
  const int hs = p.warp.n_steps - 1;
  WarpTailArgs w{A + t.out_w[hs], p.warp.steps[hs].npad, A + t.pts, A + t.warped, p.warp_type, p.warp_pivot,
                 p.warp_trans, n};
  warp_tail_kernel<<<blocks, 128, 0, s>>>(w);
  return launch_check(h, "warp_tail_kernel");
}

// compute_background_loss (training.py:118-135) and its gradient, in chunks of max_rays points.
// `warp_ids` are uint32 ids for every encoder: the reference draws them from model.warp_ids and
// hands them to warp_field.apply, so the 'time' encoder sees float(id) (training.py:121-131).
int train_background(nfb_handle* h, int P, const float* points, const unsigned* warp_ids, const float* noise,
                     float weight, cudaStream_t s) {
  using namespace nfb::train;
  const nfb::FieldProgram& p = h->prog[0];
  const nfb_config& c = h->cfg;
  const int chunk = std::min(P, h->max_rays);
  if (train_prepare_rows(h, chunk)) return -1;
  for (int p0 = 0; p0 < P; p0 += chunk) {
    const int n = std::min(chunk, P - p0);
    const TapeLayout t = tape_layout(p, n);
    float* A = h->d_tape;
    if (warp_points_forward(h, n, points + (size_t)p0 * 3, noise ? noise + (size_t)p0 * 3 : nullptr, warp_ids + p0,
                            true, s))
      return -1;
    NFB_CUDA(cudaMemsetAsync(A + t.grad_begin, 0, (size_t)(t.grad_end - t.grad_begin) * sizeof(float), s));
    NFB_CUDA(cudaMemsetAsync(h->d_dcond, 0, (size_t)n * h->cond_stride * sizeof(float), s));
    // alpha = -2, scale = 0.001: the defaults of compute_background_loss, which train_step does not override
    WarpMagArgs wm{A + t.pts, A + t.warped, nullptr, A + t.dwarped, h->d_loss + 11, -2.0f, 0.001f, weight / (float)P, n};
    warp_mag_loss_kernel<<<(unsigned)((n + 127) / 128), 128, 0, s>>>(wm);
    if (launch_check(h, "warp_mag_loss_kernel")) return -1;
    const int hs = p.warp.n_steps - 1;
    const unsigned blocks = (unsigned)((n + 127) / 128);
    WarpTailBwdArgs w{A + t.out_w[hs], p.warp.steps[hs].npad, A + t.pts, A + t.dwarped, A + t.d_out_w[hs],
                      p.warp_type, p.warp_pivot, p.warp_trans, n};
    warp_tail_bwd_kernel<<<blocks, 128, 0, s>>>(w);
    if (launch_check(h, "warp_tail_bwd_kernel")) return -1;
    if (net_backward(h, p.warp, A + t.in_w, A + t.d_in_w, t.ld_w, t.out_w, t.d_out_w, A, n, s)) return -1;
    EncodeBwdArgs e{};
    e.pts = A + t.pts; e.window = h->d_window; e.din = A + t.d_in_w; e.F = p.Fw; e.ld = t.ld_w; e.S = 1;
    e.cond_stride = h->cond_stride; e.cond_off = 0; e.n_cond = p.G; e.dpts = nullptr; e.dcond = h->d_dcond; e.rows = n;
    encode_bwd_kernel<<<blocks, 128, 0, s>>>(e);
    if (launch_check(h, "encode_bwd_kernel")) return -1;
    CondBwdArgs a{};
    a.dcond = h->d_dcond; a.stride = h->cond_stride; a.num_rays = n; a.warp_id = warp_ids + p0;
    a.d_warp_table = h->d_gwarp; a.d_app_table = h->d_gapp; a.d_cam_table = h->d_gcam;
    a.n_warp = c.num_warp_embeddings; a.n_app = c.num_appearance_embeddings; a.n_cam = c.num_camera_embeddings;
    a.G = p.G; a.A = c.num_appearance_features; a.C = c.num_camera_features; a.Fv = c.num_nerf_viewdir_freqs;
    a.use_viewdirs = c.use_viewdirs; a.use_app = c.use_appearance_metadata; a.use_cam = c.use_camera_metadata;
    a.use_trunk_c = c.use_trunk_condition; a.use_alpha_c = c.use_alpha_condition;
    set_warp_glo(h, a);
    const long long total = (long long)n * a.stride;
    cond_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(a);
    if (launch_check(h, "cond_bwd_kernel")) return -1;
    if (time_encoder_backward(h, n, warp_ids + p0, true, s)) return -1;
  }
  return 0;
}

}  // namespace

extern "C" {

int nfb_train_value_and_grad_reg(nfb_handle* h, int B, const float* origins, const float* directions,
                                 const float* viewdirs, const unsigned* warp_id, const unsigned* app_id,
                                 const unsigned* cam_id, float warp_alpha, const float* t_rand,
                                 const float* u_rand, unsigned flags, const float* rgb_target,
                                 int chunk_rays, const nfb_train_reg* reg, float* const* grads,
                                 const long long* numels, int count, float* loss_out, void* stream) {
  if (check_call(h, B)) return -1;
  if (!rgb_target || !grads || !numels || !loss_out) return fail("null argument");
  if (count != (int)h->specs.size()) return fail("expected %d gradient tensors, got %d", (int)h->specs.size(), count);
  if (flags & NFB_FLAG_METADATA_ENCODED) return fail("training with metadata_encoded=True is not supported");
  const nfb_config& c = h->cfg;
  const bool time_enc = c.warp_field_type != NFB_WARP_NONE && c.warp_metadata_encoder != NFB_WARP_ENC_GLO;
  if (time_enc && !(flags & NFB_FLAG_NO_WARP) && !warp_id)
    return fail("the 'time' / 'blend' warp metadata encoders need warp_id (metadata['time'] / ids)");
  for (int i = 0; i < count; ++i)
    if (numels[i] != h->specs[i].rows * h->specs[i].cols)
      return fail("gradient %d (%s): expected %lld elements", i, h->specs[i].name.c_str(), h->specs[i].rows * h->specs[i].cols);
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  if (B == 0) return 0;
  if (chunk_rays < 1) chunk_rays = 256;
  chunk_rays = std::min(chunk_rays, B);
  if (train_prepare(h, chunk_rays)) return -1;
  const int nc = c.num_coarse_samples, nfine = nc + c.num_fine_samples;
  const bool use_warp = !(flags & NFB_FLAG_NO_WARP);
  const bool fine = c.num_fine_samples > 0;
  if (set_window(h, warp_alpha, s)) return -1;
  NFB_CUDA(cudaMemsetAsync(h->d_gpacked, 0, (size_t)h->packed_floats * sizeof(float), s));
  NFB_CUDA(cudaMemsetAsync(h->d_gwarp, 0, (size_t)std::max(1, c.num_warp_embeddings * c.num_warp_features) * sizeof(float), s));
  NFB_CUDA(cudaMemsetAsync(h->d_gapp, 0, (size_t)std::max(1, c.num_appearance_embeddings * c.num_appearance_features) * sizeof(float), s));
  NFB_CUDA(cudaMemsetAsync(h->d_gcam, 0, (size_t)std::max(1, c.num_camera_embeddings * c.num_camera_features) * sizeof(float), s));
  NFB_CUDA(cudaMemsetAsync(h->d_loss, 0, 16 * sizeof(float), s));
  // condition vectors of the whole batch (per ray), their gradient accumulator
  if (run_cond(h, B, viewdirs ? viewdirs : directions, warp_id, app_id, cam_id, s)) return -1;
  NFB_CUDA(cudaMemsetAsync(h->d_dcond, 0, (size_t)B * h->cond_stride * sizeof(float), s));
  if (nfb_coarse_z_vals(h, B, t_rand, h->d_zc, stream)) return -1;
  const float scale = 1.f / ((float)B * 3.f);       // mean over the local batch (training.py:173)
  RegCfg rc_{};
  const RegCfg* rcfg = nullptr;
  if (reg && (reg->use_elastic_loss || reg->use_warp_reg_loss)) {
    if (!use_warp || h->prog[0].warp_type == 0)
      return fail("the elastic / warp-reg losses need a warp field (training.py:176-207)");
    if (reg->use_elastic_loss && (reg->elastic_loss_type < 0 || reg->elastic_loss_type > NFB_ELASTIC_LOG_DET))
      return fail("elastic_loss_type %d is not supported ('nr' differentiates an SVD with a repeated factor "
                  "and yields NaNs in the reference, training.py:59)", reg->elastic_loss_type);
    rc_.elastic = reg->use_elastic_loss != 0; rc_.reduce = reg->elastic_reduce_method; rc_.type = reg->elastic_loss_type;
    rc_.elastic_weight = reg->elastic_loss_weight;
    rc_.warp_reg = reg->use_warp_reg_loss != 0; rc_.warp_reg_weight = reg->warp_reg_loss_weight;
    rc_.warp_reg_alpha = reg->warp_reg_loss_alpha; rc_.warp_reg_scale = reg->warp_reg_loss_scale;
    rc_.batch_rays = B; rc_.stats = h->d_loss;
    rcfg = &rc_;
  }
  const float* cond_all = h->d_cond;
  float* dcond_all = h->d_dcond;
  for (int r0 = 0; r0 < B; r0 += chunk_rays) {
    const int R = std::min(chunk_rays, B - r0);
    // per-chunk views (the kernels index rays from 0)
    h->d_cond = const_cast<float*>(cond_all) + (size_t)r0 * h->cond_stride;
    h->d_dcond = dcond_all + (size_t)r0 * h->cond_stride;
    const float* o = origins + (size_t)r0 * 3;
    const float* d = directions + (size_t)r0 * 3;
    const float* tg = rgb_target + (size_t)r0 * 3;
    float* zc = h->d_zc + (size_t)r0 * nc;
    float* wc = h->d_tr_w;
    int rc = train_level(h, 0, R, nc, zc, o, d, tg, scale, use_warp, h->d_tr_out, wc, h->d_loss, s, rcfg);
    if (rc == 0 && fine) {
      float* zf = h->d_zf + (size_t)r0 * nfine;
      rc = run_resample(h, R, zc, wc, u_rand ? u_rand + (size_t)r0 * c.num_fine_samples : nullptr, zf, s);
      if (rc == 0)
        rc = train_level(h, 1, R, nfine, zf, o, d, tg, scale, use_warp, h->d_tr_out + 6 * (size_t)R, h->d_tr_w,
                         h->d_loss + 1, s, rcfg);
    }
    h->d_cond = const_cast<float*>(cond_all);
    h->d_dcond = dcond_all;
    if (rc) return -1;
  }
  // embedding gradients
  {
    nfb::train::CondBwdArgs a{};
    a.dcond = h->d_dcond; a.stride = h->cond_stride; a.num_rays = B;
    a.warp_id = warp_id; a.app_id = app_id; a.cam_id = cam_id;
    a.d_warp_table = h->d_gwarp; a.d_app_table = h->d_gapp; a.d_cam_table = h->d_gcam;
    a.n_warp = c.num_warp_embeddings; a.n_app = c.num_appearance_embeddings; a.n_cam = c.num_camera_embeddings;
    a.G = h->prog[0].G; a.A = c.num_appearance_features; a.C = c.num_camera_features; a.Fv = c.num_nerf_viewdir_freqs;
    a.use_viewdirs = c.use_viewdirs; a.use_app = c.use_appearance_metadata; a.use_cam = c.use_camera_metadata;
    a.use_trunk_c = c.use_trunk_condition; a.use_alpha_c = c.use_alpha_condition;
    set_warp_glo(h, a);
    const long long total = (long long)B * a.stride;
    nfb::train::cond_bwd_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(a);
    if (launch_check(h, "cond_bwd_kernel")) return -1;
  }
  if (use_warp && time_encoder_backward(h, B, warp_id, false, s)) return -1;
  // background loss (training.py:118-135, 246-257): warp_field.apply on free points
  const int P = (reg && reg->use_background_loss) ? reg->num_background_points : 0;
  if (P > 0) {
    if (!use_warp || h->prog[0].warp_type == 0) return fail("the background loss needs a warp field");
    if (!reg->background_points || !reg->background_warp_ids) return fail("background points / warp ids are null");
    if (train_background(h, P, reg->background_points, reg->background_warp_ids, reg->background_noise,
                         reg->background_loss_weight, s))
      return -1;
  }
  {
    const long long jrows = (reg && reg->use_elastic_loss) ? (reg->elastic_reduce_method == 0 ? B : (long long)B * nc) : 1;
    nfb::train::finalize_stats_kernel<<<1, 32, 0, s>>>(h->d_loss, 1.f / (float)B, 1.f / (float)jrows, P > 0 ? 1.f / (float)P : 0.f);
    if (launch_check(h, "finalize_stats_kernel")) return -1;
  }
  // packed layouts -> the caller's tensors (+=), in the order of nfb_param_info
  for (int i = 0; i < count; ++i) {
    const ParamSpec& p = h->specs[i];
    const float* base = p.table == 0 ? h->d_gpacked : p.table == 1 ? h->d_gwarp : p.table == 2 ? h->d_gapp : h->d_gcam;
    const long long n = p.rows * p.cols;
    if (n == 0) continue;
    if (!grads[i]) return fail("gradient %d (%s) is null", i, p.name.c_str());
    nfb::train::unpack_grad_kernel<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(base + p.dst_off, grads[i], p.rows, p.cols, p.ld, p.c_off);
    if (launch_check(h, "unpack_grad_kernel")) return -1;
  }
  NFB_CUDA(cudaMemcpyAsync(loss_out, h->d_loss, (reg ? 16 : 2) * sizeof(float), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int nfb_train_value_and_grad(nfb_handle* h, int B, const float* origins, const float* directions,
                             const float* viewdirs, const unsigned* warp_id, const unsigned* app_id,
                             const unsigned* cam_id, float warp_alpha, const float* t_rand,
                             const float* u_rand, unsigned flags, const float* rgb_target,
                             int chunk_rays, float* const* grads, const long long* numels, int count,
                             float* loss_out, void* stream) {
  return nfb_train_value_and_grad_reg(h, B, origins, directions, viewdirs, warp_id, app_id, cam_id, warp_alpha, t_rand,
                                      u_rand, flags, rgb_target, chunk_rays, nullptr, grads, numels, count, loss_out,
                                      stream);
}

int nfb_warp_jacobian(nfb_handle* h, int P, const float* points, const unsigned* warp_id, float warp_alpha,
                      float* warped_out, float* jacobian_out, void* stream) {
  if (!h || !points || !jacobian_out) return fail("null argument");
  if (P < 0) return fail("P must be >= 0");
  if (check_call(h, std::min(P, h->max_rays))) return -1;
  if (h->prog[0].warp_type == 0) return fail("the model has no warp field");
  cudaStream_t s = (cudaStream_t)stream;
  if (enter_stream(h, s)) return -1;
  if (P == 0) return 0;
  if (set_window(h, warp_alpha, s)) return -1;
  const int chunk = std::min(P, h->max_rays);
  if (train_prepare_rows(h, chunk)) return -1;
  for (int p0 = 0; p0 < P; p0 += chunk) {
    const int n = std::min(chunk, P - p0);
    if (warp_points_forward(h, n, points + (size_t)p0 * 3, nullptr, warp_id ? warp_id + p0 : nullptr, false, s))
      return -1;
    const nfb::FieldProgram& p = h->prog[0];
    const TapeLayout t = tape_layout(p, n);
    if (warped_out)
      NFB_CUDA(cudaMemcpyAsync(warped_out + (size_t)p0 * 3, h->d_tape + t.warped, (size_t)n * 3 * sizeof(float),
                               cudaMemcpyDeviceToDevice, s));
    if (warp_jacobian_on_tape(h, p, t, h->d_tape, nullptr, n, nullptr, nullptr, false, jacobian_out + (size_t)p0 * 9, s))
      return -1;
  }
  return 0;
}

int nfb_adam_step(float* params, const float* grads, float* m, float* v, long long n, float learning_rate,
                  float beta1, float beta2, float eps, long long step, void* stream) {
  if (!params || !grads || !m || !v) return fail("null argument");
  if (n <= 0) return 0;
  if (step < 1) return fail("adam: step counts from 1");
  const float bc1 = 1.f - powf(beta1, (float)step), bc2 = 1.f - powf(beta2, (float)step);
  nfb::train::adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(
      params, grads, m, v, n, learning_rate, beta1, beta2, eps, bc1, bc2);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail("adam_kernel launch failed: %s", cudaGetErrorString(e));
  return 0;
}

}  // extern "C"
