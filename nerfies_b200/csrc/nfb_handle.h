// Internal definition of nfb_handle and small host helpers shared by the
// translation unit's parts (nfb_api.cu, field_tc.cuh).
#pragma once
#include <cuda_runtime.h>

#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/nerfies_b200.h"
#include "common.cuh"
#include "tc_program.cuh"

namespace {

thread_local std::string g_error;

int fail(const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_error = buf;
  return -1;
}

#define NFB_CUDA(expr)                                                        \
  do {                                                                        \
    cudaError_t e_ = (expr);                                                  \
    if (e_ != cudaSuccess)                                                    \
      return fail("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_),     \
                  __FILE__, __LINE__);                                        \
  } while (0)

struct ParamSpec {
  std::string name;
  long long rows, cols;
  // destination in the packed buffer: element (r, c) -> dst_off + r * ld + c_off + c
  long long dst_off;
  int ld, c_off;
  int table;  // 0 = packed dense buffer; 1/2/3 = warp/appearance/camera table
};

__global__ void pack_kernel(const float* __restrict__ src, float* __restrict__ dst,
                            long long rows, long long cols, int ld, int c_off) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  const long long r = idx / cols, c = idx - r * cols;
  dst[r * ld + c_off + c] = src[idx];
}

int pad32(int n) { return (n + 31) / 32 * 32; }

}  // namespace

struct nfb_handle {
  nfb_config cfg;
  int max_rays = 0;
  int device = 0;
  nfb::FieldProgram prog[2];          // per level (coarse, fine)
  std::vector<ParamSpec> specs;
  long long packed_floats = 0;
  float* d_packed = nullptr;          // dense weights/biases (both levels + warp)
  float* d_warp_table = nullptr;
  float* d_app_table = nullptr;
  float* d_cam_table = nullptr;
  bool params_set = false;
  // per-model tables
  float *d_zlin = nullptr, *d_lower = nullptr, *d_upper = nullptr, *d_ulin = nullptr;
  float* d_window = nullptr;
  float h_window_alpha = NAN;
  // workspace
  float *d_cond = nullptr, *d_zc = nullptr, *d_zf = nullptr, *d_wc = nullptr;
  float* d_samples = nullptr;
  float *d_out_c = nullptr, *d_out_f = nullptr;
  // device + pinned staging for the *_host entry point
  float *d_in = nullptr, *h_in = nullptr, *h_out = nullptr;
  unsigned *d_ids = nullptr, *h_ids = nullptr;
  long long launches = 0;
  bool profiling = false;
  cudaEvent_t ev[2][2] = {{nullptr, nullptr}, {nullptr, nullptr}};
  bool ev_valid[2] = {false, false};
  int cond_stride = 0;
  int sm_count = 148;
  nfb::Net time_net{};                // TimeEncoder MLP ('time' / 'blend' warp metadata encoders)
  float time_alpha = 0.f;             // warp_extra['time_alpha'] (nfb_set_time_alpha)
  cudaStream_t last_stream = nullptr;  // stream of the previous call (see enter_stream)
  bool last_stream_valid = false;
  cudaEvent_t ev_order = nullptr;
  // training tier (train_api.cuh): tape + gradient buffers, allocated on first use
  float* d_tape = nullptr; long long tape_floats = 0;
  float *d_gpacked = nullptr, *d_gwarp = nullptr, *d_gapp = nullptr, *d_gcam = nullptr;
  float *d_dcond = nullptr, *d_tr_out = nullptr, *d_tr_w = nullptr, *d_loss = nullptr;
  float* d_ttape = nullptr; long long ttape_floats = 0;     // tangent tape (train_reg.cuh)
  int* d_sel = nullptr; long long sel_cap = 0;              // selected tape rows (median-depth samples)
  float* d_time_tape = nullptr; long long time_tape_floats = 0;   // TimeEncoder tape (train_api.cuh)
  int x3_pair_ok = -1;                // fp16x3 CTA-pair launch: -1 unknown, 0 unavailable, n = co-resident clusters
  int debug_bits = 0;                 // FieldArgs::debug bits set through the test hook (abort-path test)
  long long* trace = nullptr;
  int trace_cap = 0;
  // tensor-core path (precision != fp32)
  nfb::tc::TcProgram tcprog[2];
  nfb::tc::TcBias tcbias[2];          // host copy of the per-step biases (kernel parameter)
  nfb::tc::X3Consts x3c[2];           // fp16x3 mode: biases + alpha head (kernel parameter)
  unsigned char* d_wpack = nullptr;   // bf16 weight units, shared-memory image
  float* d_aux = nullptr;             // fp32 biases + alpha head
  long long wpack_bytes = 0, aux_floats = 0;
  struct TcPackJob { int level, step, chunk; int simt_w_off, ld, n, n0, k_total; std::vector<int> k_map;
                     std::vector<int> unit_pos; };   // fp16x3: issue-order position of each K-block's unit within the step
  std::vector<TcPackJob> tc_jobs;
  struct TcAuxJob { int src_off, count, stride, dst_off; };
  std::vector<TcAuxJob> tc_aux_jobs;
};

