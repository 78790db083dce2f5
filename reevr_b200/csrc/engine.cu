// engine.cu — host side of the B200 partitioned-convolution engine + the C ABI (include/b200conv.h).
//
// One handle = C mono convolvers sharing a stage schedule.  Stage s = uniform partitioned
// convolver with block B_s over the IR taps [off_s, off_{s+1}) whose contribution is delayed by
// q_s = off_s / B_s blocks (the scheme TwoStageFFTConvolver.cpp:120-138,166-222 uses for its
// tails, generalised): stage 0 is the zero-latency head (handles partially filled blocks like
// FFTConvolver.cpp:164-193), stages >= 1 work on completed blocks only and deposit their
// output into a look-ahead ring the head's inverse-FFT epilogue adds on top.
//
// Device state per stage (all float32 / float2, resident for the handle's lifetime):
//   H   [C][Prows][B]   IR partition spectra (this shard's partition range), zero padded
//   X   [C][R][B]       input-spectrum timeline = the frequency-domain delay line, linear:
//                       row `head` is the open block; partition p of output block t reads row
//                       head + t - p.  Compacted (history moved to the front) when full.
//   Y[2] [1+T][C][B]    spectra of the current launch group (double-buffered by group so that reduce +
//                       inverse FFT of group i overlap the sweep of group i+1); row 0 = last completed
//                       block of the previous group (the overlap state, FFTConvolver.cpp:204 kept in
//                       the frequency domain)
//   inbuf [C][B + Lmax] time-domain input of the open block + this call's samples
//   fut [C][ring]       (stages >= 1) look-ahead output ring, indexed by absolute position
// Streams: s_main (forward FFT + sweep), s_post (exchange/reduce + inverse FFT + mixdown), s_in / s_out
// (PCIe copies of the pipelined host path).  Multi-GPU: partition-range shards with either a reduce hook
// (NCCL) or the fused slot exchange over peer memory (run_group_p2p).
#if defined(PC_EMULATE)
#include "cuda_emu.h"      // tests/emu: host stand-in for the CUDA runtime (test infrastructure)
#else
#include <cuda_runtime.h>
#endif

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "../../include/b200conv.h"
#include "kernels.cuh"
#include "kernels_stream.cuh"
#include "kernels_fft512.cuh"
#include "kernels_rt.cuh"
#include "kernels_chain.cuh"
#include "kernels_tfft.cuh"
#if !defined(PC_EMULATE)
#include "kernels_tc.cuh"
#endif

namespace {

constexpr int kDPre = 8;          // max prefetch distance of the CMAC kernels (rows readable past the end)
constexpr int kPadP = 96;         // H / history rows are padded to a multiple of this = lcm of every sweep tile height TT in use (8, 12, 16, 24, 32)
constexpr int kMaxTT = 32;        // slack rows after the newest X row
constexpr int kDefaultBatch = 4736;   // 148 SMs * 32
constexpr int kMaxBlockLog2 = 13;     // B <= 8192 (two M-point ping-pong buffers = 128 KB smem)

inline size_t next_pow2(size_t v) { size_t p = 1; while (p < v) p *= 2; return p; }
inline int round_up(int v, int m) { return (v + m - 1) / m * m; }

struct Stage {
  int B = 0;
  size_t tap_off = 0;      // first IR tap of this stage
  size_t tap_end = 0;      // one past the last tap (over all channels)
  int q = 0;               // output delay in blocks (tap_off / B)
  int P_full = 0;          // partitions of the stage (max over channels)
  int p_begin = 0, p_end = 0;   // this shard's partition range
  int P = 0;               // p_end - p_begin
  int Prows = 0;           // allocated H rows
  int hist = 0;            // X rows kept before the open block
  int Tcap = 0;            // max blocks per launch group
  int R = 0;               // X rows allocated
  long long head = 0;      // X row of the open block
  long long blocks_done = 0;   // completed blocks since init/clear
  int fill = 0;            // samples of the open block already buffered
  float2* H = nullptr;
  float2* X = nullptr;
  float2* Y[2] = {nullptr, nullptr};   // double buffer: the sweep of group i+1 may overlap reduce+IFFT of group i
  int ybuf = 0;
  cudaEvent_t ev_sweep[2] = {nullptr, nullptr};   // Y[b] rows written by the sweep
  cudaEvent_t ev_post[2] = {nullptr, nullptr};    // Y[b] no longer needed by reduce / inverse FFT
  float2* tw = nullptr;
  float2* tab512 = nullptr;   // B == 512: tables of the register-resident FFT kernels
  float* inbuf = nullptr;           // open block of this stage (+ the current call's samples on the batch path)
  float* inbuf_alt = nullptr;       // stages >= 1: second buffer — a tail block enqueued on s_tail keeps reading the
                                    // one it completed while the following calls already fill the other
  size_t in_stride = 0;
  // tail blocks enqueued on the low-priority stream by the real-time path (stages >= 1)
  cudaEvent_t ev_job[2] = {nullptr, nullptr};
  long long job_out_start[2] = {0, 0};   // absolute sample position where the job's output is first needed
  bool job_waited[2] = {true, true};
  unsigned long long njobs = 0;
  float* fut = nullptr;
  size_t ring = 0;
};

struct EventPair { cudaEvent_t a, b; int kind; };

}  // namespace

struct b200conv {
  b200conv_config cfg{};
  int C = 1;
  std::string err;
  bool sticky_cuda_error = false;
  std::vector<Stage> stages;
  std::vector<size_t> ir_len;     // post-trim
  size_t Lmax = 0;                // max samples per launch group
  long long abs_pos = 0;          // absolute stream position (samples since init/clear)
  cudaStream_t s_main = nullptr, s_post = nullptr, s_in = nullptr, s_out = nullptr;
  cudaStream_t s_tail = nullptr;     // lowest priority: tail-stage blocks of the real-time path (run_tail_block)
  cudaStream_t s_launch = nullptr;   // stream the kernel launchers use: s_main, or s_tail while a tail block is enqueued
  cudaEvent_t ev_rt = nullptr;       // real-time kernel of the current call done (s_main)
  float* hpin_in_dev = nullptr;      // device-side addresses of the pinned staging buffers (zero-copy I/O)
  float* hpin_out_dev = nullptr;
  unsigned long long* stream_ticket = nullptr;   // ticket counters of the dynamic streaming sweep (device, 256 words)
  unsigned long long stream_ticket_base = 0;
  unsigned int stream_launches = 0;             // alternates the walk direction of the streaming sweep
  bool opt_stream_alt = std::getenv("B200CONV_NO_STREAM_ALT") == nullptr;
  unsigned int* hflag = nullptr;     // pinned completion word of the real-time kernel (+ its device-side address)
  unsigned int* hflag_dev = nullptr;
  unsigned int flag_epoch = 0;
  cudaEvent_t ev_h2d[2]{}, ev_comp[2]{}, ev_d2h[2]{}, ev_din[2]{};
  cudaEvent_t ev_join = nullptr;
  float* din[2] = {nullptr, nullptr};
  float* dout[2] = {nullptr, nullptr};
  float* hpin_in = nullptr;       // pinned host staging of the latency path: all channels of a call in ONE copy
  float* hpin_out = nullptr;
  size_t hpin_cap = 0;            // samples per channel the staging holds
  unsigned long long launches = 0;
  // timing
  bool timing = false;
  std::vector<EventPair> ev_pool;
  size_t ev_used = 0;
  float t_cmac = 0, t_fft = 0, t_ifft = 0;
  int n_cmac = 0;
  // sharding
  b200conv_reduce_fn reduce = nullptr;
  void* reduce_user = nullptr;
  int n_sm = 148;
  // I/O routing + mixdown (b200conv_set_routing)
  bool route_on = false;
  int n_in = 0, n_out = 0;
  int in_map[8] = {};
  float mix[64] = {};
  float* dch[1] = {nullptr};                // per-convolver outputs [C][Lmax] before the mixdown
  // time-slice sharding: Y row 0 (the overlap state, spectrum of the last completed block) does not belong to
  // the block in front of the open one any more (the timeline was advanced by forward FFTs only)
  bool yprev_stale = false;
  // send / wet chain around the convolver (b200conv_chain_*, kernels_chain.cuh)
  bool chain_on = false;
  bool route_in_only = false;        // chain calls: convolver c reads chain input c & 1, outputs stay per convolver
  b200conv_chain_config chain_cfg{};
  pc::ChainFilter chain_lc{}, chain_hc{};
  float* c_io = nullptr;             // [dry L, dry R, ysend, yrev, out L, out R][Lmax] staging
  float* c_conv_in = nullptr;        // [2][Lmax] convolver input (after filters + predelay)
  float* c_filt = nullptr;           // [2][Lmax]
  float* c_state = nullptr;          // [2][8] filter states
  float* c_hpin = nullptr;           // pinned [dry L, dry R, ysend, yrev, out L, out R][hpin_cap]: zero-copy I/O of real-time chain calls
  float* c_hpin_dev = nullptr;
  float* c_ring = nullptr;           // [2][ring] predelay ring
  size_t c_ring_size = 0;
  long long c_ring_pos = 0;
  // b200conv_init_*_shaped: the taps handed to init are DEVICE buffers (shaped there) with known post-trim lengths
  bool ir_on_device = false;
  const size_t* ir_trimmed = nullptr;
  // tuning / A-B switches (b200conv_set_option; defaults from the environment)
  bool opt_rt = std::getenv("B200CONV_NO_RT") == nullptr;
  bool opt_fft512 = std::getenv("B200CONV_NO_FFT512") == nullptr;
  bool opt_slice_tail = true;        // sliced calls: also transform the last P blocks of the call (full-state contract)
  // tensor-core sweep (kernels_tc.cuh): Toeplitz tile images of one stage's H, per-bin time lines, partial planes
  bool opt_tc = std::getenv("B200CONV_NO_TC") == nullptr;
  float* tc_A = nullptr;
  const void* tc_A_for = nullptr;    // H the images were built from (+ its geometry)
  int tc_A_P = 0, tc_A_B = 0, tc_A_C = 0;
  float* tc_Xt = nullptr;
  float* tc_Yt = nullptr;
  size_t tc_A_bytes = 0, tc_Xt_bytes = 0, tc_Yt_bytes = 0;
  int* tc_err = nullptr;             // mapped pinned word: a barrier wait of k_tc_sweep gave up
  int* tc_err_dev = nullptr;
  bool tc_attr_set = false;
  bool tc_alloc_failed = false;      // the scratch did not fit once: stay on the FFMA sweep
  // FFT sweep along the block axis (kernels_tfft.cuh): filter spectra of one stage's H, twiddles of the length-N transform
  bool opt_tfft = std::getenv("B200CONV_NO_TFFT") == nullptr;
  float2* tfft_Hf = nullptr;
  size_t tfft_Hf_bytes = 0;
  const void* tfft_Hf_for = nullptr;   // H the spectra were built from (+ its geometry)
  int tfft_Hf_P = 0, tfft_Hf_B = 0, tfft_Hf_C = 0, tfft_Hf_N = 0;
  float2* tfft_tw = nullptr;
  size_t tfft_tw_bytes = 0;
  int tfft_tw_N = 0;
  bool tfft_attr_set[3] = {false, false, false};
  bool tfft_alloc_failed = false;    // the spectra did not fit once: stay on the other sweeps
  int last_variant = 0;              // sweep form the last launch_cmac resolved to (b200conv_last_sweep_variant)
  // slot exchange (fused multi-GPU path), stage 0 of a single-stage handle
  bool p2p_on = false;
  int p2p_mode = 0;
  int xSR = 0;                       // rows per slot (slice rows + halo + spare)
  size_t xslot = 0;                  // float2 per slot
  float2* Yx[2] = {nullptr, nullptr};       // [G slots][xSR][C][B]
  float2* Hh = nullptr;                     // [3][G][C][B] halo of the next group's first slice (owner 0)
  float* xout[2] = {nullptr, nullptr};      // [C][Lmax] output exchange (used on shard 0)
  unsigned int* xflags = nullptr;           // 8 barrier words + 1 error word
  int hidx = 0;                             // halo buffer in use (mod 3)
  unsigned int bar_epoch = 0;
  float2* peerYx[8][2] = {};
  float2* peerHh0 = nullptr;
  float* peer_xout0[2] = {nullptr, nullptr};
  unsigned int* peer_flags[8] = {};
  bool bcast_in = false;                    // shard 0 uploads the input and stores it into the peers' staging (NVLink)
  float* peer_din[8][2] = {};               // every shard's din[0..1] (mapped on shard 0 when the broadcast is enabled)
  std::vector<unsigned char> din_records;   // the peers' exported din records, opened lazily
  unsigned int in_epoch = 0;                // epoch of the "input landed" barrier (flag words 16..23)
  unsigned long long xgrp = 0;              // slot-exchange groups issued so far
  cudaEvent_t ev_b1[2] = {nullptr, nullptr};   // first barrier of group (xgrp & 1) passed: peers finished reading din
  std::vector<void*> ipc_opened;
  b200conv_barrier_fn host_barrier = nullptr;
  void* host_barrier_user = nullptr;
};

namespace {

// Only errors that poison the CUDA context (or mean there is no usable device) make the handle fail for
// good; everything else — out of memory while loading a long IR, CUDA IPC not permitted in this container,
// an invalid argument — is cleared from the runtime, reported through the status code and leaves the
// handle usable (the caller can fall back to the reduce hook, load a shorter IR, ...).
bool cuda_error_is_sticky(cudaError_t e) {
#if defined(PC_EMULATE)
  (void)e;
  return false;
#else
  switch (e) {
    case cudaErrorIllegalAddress: case cudaErrorLaunchFailure: case cudaErrorLaunchTimeout:
    case cudaErrorIllegalInstruction: case cudaErrorMisalignedAddress: case cudaErrorInvalidAddressSpace:
    case cudaErrorInvalidPc: case cudaErrorHardwareStackError: case cudaErrorAssert:
    case cudaErrorECCUncorrectable: case cudaErrorNoDevice: case cudaErrorInsufficientDriver:
    case cudaErrorDevicesUnavailable: case cudaErrorCudartUnloading: case cudaErrorUnknown:
      return true;
    default:
      return false;
  }
#endif
}

int cuda_fail(b200conv* h, cudaError_t e, const char* what) {
  h->err = std::string(what) + ": " + cudaGetErrorString(e);
  cudaGetLastError();                                   // clear the runtime's (non-sticky) last error
  if (cuda_error_is_sticky(e)) h->sticky_cuda_error = true;
  return e == cudaErrorMemoryAllocation ? B200CONV_ENOMEM : B200CONV_ECUDA;
}

#define CU_CHECK(h, expr)                                                                  \
  do {                                                                                     \
    cudaError_t e__ = (expr);                                                              \
    if (e__ != cudaSuccess) return cuda_fail((h), e__, #expr);                             \
  } while (0)

int fail(b200conv* h, int code, const std::string& msg) { h->err = msg; return code; }

void free_stage(Stage& s) {
  cudaFree(s.H); cudaFree(s.X); cudaFree(s.Y[0]); cudaFree(s.Y[1]); cudaFree(s.tw); cudaFree(s.tab512); cudaFree(s.inbuf); cudaFree(s.inbuf_alt); cudaFree(s.fut);
  for (int i = 0; i < 2; ++i) {
    if (s.ev_job[i]) cudaEventDestroy(s.ev_job[i]);
    if (s.ev_sweep[i]) cudaEventDestroy(s.ev_sweep[i]);
    if (s.ev_post[i]) cudaEventDestroy(s.ev_post[i]);
  }
  s = Stage();
}

void p2p_release(b200conv* h) {
#if !defined(PC_EMULATE)
  for (void* p : h->ipc_opened) cudaIpcCloseMemHandle(p);
#endif
  h->ipc_opened.clear();
  cudaFree(h->Yx[0]); cudaFree(h->Yx[1]); cudaFree(h->Hh); cudaFree(h->xout[0]); cudaFree(h->xout[1]); cudaFree(h->xflags);
  h->Yx[0] = h->Yx[1] = nullptr; h->Hh = nullptr; h->xout[0] = h->xout[1] = nullptr; h->xflags = nullptr;
  h->p2p_on = false; h->hidx = 0; h->bar_epoch = 0; h->in_epoch = 0; h->xgrp = 0; h->bcast_in = false;
  for (int i = 0; i < 2; ++i) { if (h->ev_b1[i]) cudaEventDestroy(h->ev_b1[i]); h->ev_b1[i] = nullptr; }
}

void free_all(b200conv* h) {
  p2p_release(h);
  for (auto& s : h->stages) free_stage(s);
  h->stages.clear();
  for (int i = 0; i < 2; ++i) {
    cudaFree(h->din[i]); cudaFree(h->dout[i]);
    h->din[i] = h->dout[i] = nullptr;
  }
  cudaFree(h->dch[0]); h->dch[0] = nullptr;
  cudaFree(h->tc_A); cudaFree(h->tc_Xt); cudaFree(h->tc_Yt);
  h->tc_A = h->tc_Xt = h->tc_Yt = nullptr; h->tc_A_for = nullptr; h->tc_A_bytes = h->tc_Xt_bytes = h->tc_Yt_bytes = 0;
  if (h->tc_err) cudaFreeHost(h->tc_err);
  h->tc_err = h->tc_err_dev = nullptr; h->tc_alloc_failed = false;
  cudaFree(h->tfft_Hf); cudaFree(h->tfft_tw);
  h->tfft_Hf = h->tfft_tw = nullptr; h->tfft_Hf_for = nullptr; h->tfft_Hf_bytes = h->tfft_tw_bytes = 0; h->tfft_tw_N = 0;
  h->tfft_alloc_failed = false;
  cudaFree(h->c_io); cudaFree(h->c_conv_in); cudaFree(h->c_filt); cudaFree(h->c_state); cudaFree(h->c_ring);
  if (h->c_hpin) cudaFreeHost(h->c_hpin);
  h->c_hpin = h->c_hpin_dev = nullptr;
  h->c_io = h->c_conv_in = h->c_filt = h->c_state = h->c_ring = nullptr;
  h->c_ring_size = 0; h->c_ring_pos = 0;
  h->chain_on = false; h->route_in_only = false;
  if (h->hpin_in) cudaFreeHost(h->hpin_in);
  if (h->hpin_out) cudaFreeHost(h->hpin_out);
  if (h->hflag) cudaFreeHost(h->hflag);
  h->hflag = h->hflag_dev = nullptr;
  h->hpin_in = h->hpin_out = nullptr; h->hpin_cap = 0;
  h->hpin_in_dev = h->hpin_out_dev = nullptr;
  h->ir_len.assign(h->C, 0);
  h->abs_pos = 0;
  h->Lmax = 0;
}

// ---- timing helpers ------------------------------------------------------------------------
enum { kKindFft = 0, kKindCmac = 1, kKindIfft = 2 };

int timing_begin(b200conv* h, int kind, cudaStream_t st = nullptr) {
  if (!st) st = h->s_launch;
  if (!h->timing) return -1;
  if (h->ev_used == h->ev_pool.size()) {
    EventPair p;
    if (cudaEventCreate(&p.a) != cudaSuccess || cudaEventCreate(&p.b) != cudaSuccess) return -1;
    h->ev_pool.push_back(p);
  }
  int id = (int)h->ev_used++;
  h->ev_pool[id].kind = kind;
  cudaEventRecord(h->ev_pool[id].a, st);
  return id;
}
void timing_end(b200conv* h, int id, cudaStream_t st = nullptr) {
  if (id >= 0) cudaEventRecord(h->ev_pool[id].b, st ? st : h->s_launch);
}
void timing_collect(b200conv* h) {
  h->t_cmac = h->t_fft = h->t_ifft = 0;
  h->n_cmac = 0;
  for (size_t i = 0; i < h->ev_used; ++i) {
    float ms = 0;
    if (cudaEventElapsedTime(&ms, h->ev_pool[i].a, h->ev_pool[i].b) != cudaSuccess) continue;
    if (h->ev_pool[i].kind == kKindCmac) { h->t_cmac += ms; h->n_cmac++; }
    else if (h->ev_pool[i].kind == kKindFft) h->t_fft += ms;
    else h->t_ifft += ms;
  }
}

// twiddle table of the M-point transforms (layout: kernels.cuh tw_pass_offset), computed in double
std::vector<float2> fft_twiddles(int M) {
  std::vector<float2> tw(pc::tw_table_len(M));
  for (int k = 0; k <= M / 2; ++k) {                       // split twiddles exp(-2*pi*i*k/(2M))
    const double a = -2.0 * M_PI * (double)k / (2.0 * (double)M);
    tw[k] = make_float2((float)std::cos(a), (float)std::sin(a));
  }
  for (int p = 1; p < M;) {                                // pass twiddles exp(-2*pi*i*r*k/(p*R))
    const int R = pc::pass_radix(M, p);
    const int off = pc::tw_pass_offset(M, p);
    for (int r = 1; r < R; ++r)
      for (int k = 0; k < p; ++k) {
        const double a = -2.0 * M_PI * (double)r * (double)k / ((double)p * (double)R);
        tw[off + (r - 1) * p + k] = make_float2((float)std::cos(a), (float)std::sin(a));
      }
    p *= R;
  }
  return tw;
}

// ---- kernel launchers ----------------------------------------------------------------------
// block (NT, ty): NT threads per transform, ty transforms per CTA; see k_fwd_fft
struct FftGeom { dim3 grid, block; size_t smem; bool tws; };

FftGeom fft_geometry(int M, int nblocks, int C) {
  FftGeom g;
  const int nt = pc::fft_threads(M);
  int ty = 1;
  if (pc::fft_warp_mode(M)) {            // one warp per transform
    ty = std::max(1, std::min(8, 4096 / std::max(M, 1)));
    ty = std::min(ty, std::max(1, nblocks));
    g.tws = (long long)nblocks * C >= 64;    // real-time calls: a few transforms, table read through L1 instead
  } else {
    g.tws = (M <= 4096);
  }
  g.block = dim3(nt, ty, 1);
  g.grid = dim3((nblocks + ty - 1) / ty, C, 1);
  const size_t tl = g.tws ? (((size_t)pc::tw_table_len(M) + 15) & ~(size_t)15) : 0;
  g.smem = (tl + (size_t)ty * 2 * std::max(M, 16)) * sizeof(float2);
  return g;
}

#if !defined(PC_EMULATE)
template <int L>
void launch_fwd_l(const pc::FwdParams& P, const FftGeom& g, cudaStream_t st) {
  if (g.tws) pc::k_fwd_fft<(1 << L), true><<<g.grid, g.block, g.smem, st>>>(P);
  else pc::k_fwd_fft<(1 << L), false><<<g.grid, g.block, g.smem, st>>>(P);
}
template <int L>
void launch_inv_l(const pc::InvParams& P, const FftGeom& g, cudaStream_t st) {
  if (P.n_partials > 1) {
    if (g.tws) pc::k_inv_fft_ola<(1 << L), true, true><<<g.grid, g.block, g.smem, st>>>(P);
    else pc::k_inv_fft_ola<(1 << L), false, true><<<g.grid, g.block, g.smem, st>>>(P);
  } else {
    if (g.tws) pc::k_inv_fft_ola<(1 << L), true, false><<<g.grid, g.block, g.smem, st>>>(P);
    else pc::k_inv_fft_ola<(1 << L), false, false><<<g.grid, g.block, g.smem, st>>>(P);
  }
}
template <int L>
bool fft_set_smem_attr() {
  const int kSmem = 200 * 1024;   // B = 4096: 48 KB table + 64 KB ping-pong buffers; B = 8192: 128 KB buffers
  bool ok = cudaFuncSetAttribute(pc::k_fwd_fft<(1 << L), true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_fwd_fft<(1 << L), false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_inv_fft_ola<(1 << L), true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_inv_fft_ola<(1 << L), false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_inv_fft_ola<(1 << L), true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_inv_fft_ola<(1 << L), false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem) == cudaSuccess;
  return ok;
}
bool stream_set_smem_attr() {
  bool ok = true;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 2 * pc::kStreamStageBytes + 64) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 4 * pc::kStreamStageBytes + 64) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 6 * pc::kStreamStageBytes + 128) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 12 * pc::kStreamStageBytes + 256) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma_dyn<6>, cudaFuncAttributeMaxDynamicSharedMemorySize, 6 * pc::kStreamStageBytes + 256) == cudaSuccess;
  ok = ok && cudaFuncSetAttribute(pc::k_cmac_stream_tma_dyn<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, 12 * pc::kStreamStageBytes + 512) == cudaSuccess;
  return ok;
}
#define PC_FOR_EACH_LOG2(X) X(0) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(9) X(10) X(11) X(12) X(13)
#endif

// register-resident kernels for B = 512 (kernels_fft512.cuh): batches only — a real-time call of a few transforms
// would pay the per-CTA table staging for nothing
constexpr int kF512MinTransforms = 32;
constexpr size_t kF512Smem = (size_t)(pc::kF512_TabLen + 8 * pc::kF512_Xch) * sizeof(float2);

bool use_fft512(const b200conv* h, int M, int nblocks, int C, const float2* tab) {
  return h->opt_fft512 && M == pc::kF512_M && tab != nullptr && (long long)nblocks * C >= kF512MinTransforms;
}

int launch_fwd(b200conv* h, const pc::FwdParams& P, int C) {
  if (use_fft512(h, P.M, P.nblocks, C, P.tab512)) {
    int id = timing_begin(h, kKindFft);
#if defined(PC_EMULATE)
    pc::emu_fwd_fft512(P.nblocks, C, P, P.tab512);
#else
    const int gx = std::max(1, std::min((P.nblocks + 7) / 8, (4 * h->n_sm + C - 1) / C));
    pc::k_fwd_fft512<<<dim3(gx, C, 1), dim3(32, 8, 1), kF512Smem, h->s_launch>>>(P, P.tab512);
#endif
    timing_end(h, id);
    h->launches++;
    CU_CHECK(h, cudaGetLastError());
    return 0;
  }
  const FftGeom g = fft_geometry(P.M, P.nblocks, C);
  int id = timing_begin(h, kKindFft);
#if defined(PC_EMULATE)
  pc::emu_fwd_fft({(int)g.grid.x, (int)g.grid.y, 1}, {(int)g.block.x, (int)g.block.y, 1}, P);
#else
  switch (pc::ilog2(P.M)) {
#define PC_CASE(L) case L: launch_fwd_l<L>(P, g, h->s_launch); break;
    PC_FOR_EACH_LOG2(PC_CASE)
#undef PC_CASE
    default: return fail(h, B200CONV_EINVAL, "unsupported transform size");
  }
#endif
  timing_end(h, id);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

int launch_inv(b200conv* h, const pc::InvParams& P, int C, cudaStream_t st) {
  if (P.n_partials <= 1 && use_fft512(h, P.M, P.nblocks, C, P.tab512)) {
    // whole blocks inside the destination, nothing added on top, linear and 8-byte aligned: float2 stores
    const bool fast = P.n_add == 0 && P.mask == -1 && P.lo <= P.index0 && P.hi >= P.index0 + (long long)P.nblocks * P.M &&
                      (P.index0 & 1) == 0 && (P.dst_cstride & 1) == 0 && (reinterpret_cast<size_t>(P.dst) & 7) == 0;
    int id = timing_begin(h, kKindIfft, st);
#if defined(PC_EMULATE)
    pc::emu_inv_fft512(P.nblocks, C, P, P.tab512, fast);
#else
    const int gx = std::max(1, std::min((P.nblocks + 7) / 8, (3 * h->n_sm + C - 1) / C));
    if (fast) pc::k_inv_fft512<true><<<dim3(gx, C, 1), dim3(32, 8, 1), kF512Smem, st>>>(P, P.tab512);
    else pc::k_inv_fft512<false><<<dim3(gx, C, 1), dim3(32, 8, 1), kF512Smem, st>>>(P, P.tab512);
#endif
    timing_end(h, id, st);
    h->launches++;
    CU_CHECK(h, cudaGetLastError());
    return 0;
  }
  const FftGeom g = fft_geometry(P.M, P.nblocks, C);
  int id = timing_begin(h, kKindIfft, st);
#if defined(PC_EMULATE)
  pc::emu_inv_fft_ola({(int)g.grid.x, (int)g.grid.y, 1}, {(int)g.block.x, (int)g.block.y, 1}, P);
#else
  switch (pc::ilog2(P.M)) {
#define PC_CASE(L) case L: launch_inv_l<L>(P, g, st); break;
    PC_FOR_EACH_LOG2(PC_CASE)
#undef PC_CASE
    default: return fail(h, B200CONV_EINVAL, "unsupported transform size");
  }
#endif
  timing_end(h, id, st);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

template <int TT, int D, int TW, int BS = 0>
void launch_cmac_t(b200conv* h, pc::CmacParams P, int C) {
  P.Ppad = round_up(P.Ppad, TT);
  dim3 block(32, TW, 1);
  dim3 grid((P.B + 31) / 32, (P.nblocks + TT * TW - 1) / (TT * TW), C);
#if defined(PC_EMULATE)
  (void)block;
  pc::emu_cmac_batch<TT, D, TW>({(int)grid.x, (int)grid.y, (int)grid.z}, P);
#else
  pc::k_cmac_batch<TT, D, TW, BS><<<grid, block, 0, h->s_launch>>>(P);
#endif
}

template <int TT, int D, int TW, int BS, int MINB>
void launch_cmac2_t(b200conv* h, pc::CmacParams P, int C) {
  P.Ppad = round_up(P.Ppad, TT);
  dim3 block(32, TW, 1);
  dim3 grid((P.B + 31) / 32, (P.nblocks + TT * TW - 1) / (TT * TW), C);
#if defined(PC_EMULATE)
  (void)block;
  pc::emu_cmac_batch2<TT, D, TW>({(int)grid.x, (int)grid.y, (int)grid.z}, P);
#else
  pc::k_cmac_batch2<TT, D, TW, BS, MINB><<<grid, block, 0, h->s_launch>>>(P);
#endif
}

template <int TT, int D, int TW, int MINB>
void launch_cmac2_bs(b200conv* h, const pc::CmacParams& P, int C) {
  switch (P.B) {
    case 128: launch_cmac2_t<TT, D, TW, 128, MINB>(h, P, C); break;
    case 512: launch_cmac2_t<TT, D, TW, 512, MINB>(h, P, C); break;
    case 8192: launch_cmac2_t<TT, D, TW, 8192, MINB>(h, P, C); break;
    default: launch_cmac2_t<TT, D, TW, 0, MINB>(h, P, C); break;
  }
}

// compile-time row pitch for the common block sizes (immediate load offsets), runtime pitch otherwise
template <int TT, int D, int TW>
void launch_cmac_bs(b200conv* h, const pc::CmacParams& P, int C) {
  switch (P.B) {
    case 128: launch_cmac_t<TT, D, TW, 128>(h, P, C); break;
    case 512: launch_cmac_t<TT, D, TW, 512>(h, P, C); break;
    case 8192: launch_cmac_t<TT, D, TW, 8192>(h, P, C); break;
    default: launch_cmac_t<TT, D, TW, 0>(h, P, C); break;
  }
}

constexpr int kStreamNBS = 4;      // blocks per launch the streaming sweep handles
constexpr int kStreamPW = 8;       // warps per CTA, each striding over the CTA's partition slice

int launch_cmac_stream(b200conv* h, const pc::CmacParams& P, int C) {
  pc::StreamParams S{};
  S.H = P.H; S.h_cstride = P.h_cstride;
  S.X = P.X; S.x_cstride = P.x_cstride; S.xrow0 = P.xrow0;
  S.Y = P.Y; S.y_cstride = P.y_cstride; S.y_rstride = P.y_rstride; S.yrow0 = P.yrow0;
  S.B = P.B; S.P = P.Ppad; S.nblocks = P.nblocks;
  const int ktiles = (P.B / 2 + 31) / 32;
  // enough CTAs for ~2 per SM, but at least kStreamPW*4 partitions per CTA
  int nsplit = std::max(1, (2 * h->n_sm) / std::max(1, ktiles * C));
  nsplit = std::max(1, std::min(nsplit, P.Ppad / (kStreamPW * 4)));
  S.nsplit = nsplit;
  if (nsplit > 1) {
    // rows [yrow0, yrow0+nb) of every channel are contiguous (row pitch C*B)
    CU_CHECK(h, cudaMemsetAsync(S.Y + S.yrow0 * S.y_rstride, 0, (size_t)P.nblocks * S.y_rstride * sizeof(float2), h->s_launch));
  }
  dim3 grid(ktiles, nsplit, C), block(32, kStreamPW, 1);
  int id = timing_begin(h, kKindCmac);
#if defined(PC_EMULATE)
  (void)block;
  pc::emu_cmac_stream<kStreamNBS, kStreamPW>({(int)grid.x, (int)grid.y, (int)grid.z}, S);
#else
  pc::k_cmac_stream<kStreamNBS, kStreamPW><<<grid, block, 0, h->s_launch>>>(S);
#endif
  timing_end(h, id);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

template <int NB, int U>
void launch_stream_rows_t(b200conv* h, const pc::StreamParams& S, dim3 grid, int threads) {
#if defined(PC_EMULATE)
  pc::emu_cmac_stream_rows<NB, U>({(int)grid.x, (int)grid.y, (int)grid.z}, threads, S);
#else
  pc::k_cmac_stream_rows<NB, U><<<grid, dim3(threads, 1, 1), 0, h->s_launch>>>(S);
#endif
}

// row-walking streaming sweep (B >= 64): see k_cmac_stream_rows
int launch_cmac_stream_rows(b200conv* h, const pc::CmacParams& P, int C) {
  pc::StreamParams S{};
  S.H = P.H; S.h_cstride = P.h_cstride;
  S.X = P.X; S.x_cstride = P.x_cstride; S.xrow0 = P.xrow0;
  S.Y = P.Y; S.y_cstride = P.y_cstride; S.y_rstride = P.y_rstride; S.yrow0 = P.yrow0;
  S.B = P.B; S.P = P.Ppad; S.nblocks = P.nblocks;
  const int threads = std::min(256, P.B / 2);
  const int xt = (P.B / 2 + threads - 1) / threads;
  // ~3 CTAs per SM, but no CTA with fewer than 8 partitions (one unrolled load batch)
  int nsplit = std::max(1, (3 * h->n_sm) / std::max(1, xt * C));
  nsplit = std::max(1, std::min(nsplit, std::max(1, P.Ppad / 8)));
  S.nsplit = nsplit;
  if (nsplit > 1)
    CU_CHECK(h, cudaMemsetAsync(S.Y + S.yrow0 * S.y_rstride, 0, (size_t)P.nblocks * S.y_rstride * sizeof(float2), h->s_launch));
  dim3 grid(xt, nsplit, C);
  int id = timing_begin(h, kKindCmac);
  if (P.nblocks <= 1) launch_stream_rows_t<1, 8>(h, S, grid, threads);
  else if (P.nblocks == 2) launch_stream_rows_t<2, 4>(h, S, grid, threads);
  else launch_stream_rows_t<4, 2>(h, S, grid, threads);
  timing_end(h, id);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

// TMA-fed streaming sweep (one block per launch, B >= 64): see kernels_stream.cuh.  S ring stages of 16 KB per
// CTA, `per_sm` CTAs per SM (S * per_sm * 16 KB <= 192 KB of shared memory per SM in flight).
template <int S>
int launch_stream_tma_dyn_s(b200conv* h, const pc::StreamParams& S_, dim3 grid) {
#if defined(PC_EMULATE)
  pc::emu_cmac_stream_tma_dyn({(int)grid.x, (int)grid.y, (int)grid.z}, S_);
#else
  const size_t smem = (size_t)S * pc::kStreamStageBytes + 16 * S + 8 * S;
  pc::k_cmac_stream_tma_dyn<S><<<grid, dim3(288, 1, 1), smem, h->s_launch>>>(S_);
#endif
  return 0;
}

template <int S>
int launch_stream_tma_s(b200conv* h, const pc::StreamParams& S_, dim3 grid) {
#if defined(PC_EMULATE)
  pc::emu_cmac_stream_tma({(int)grid.x, (int)grid.y, (int)grid.z}, S_);
#else
  const size_t smem = (size_t)S * pc::kStreamStageBytes + 16 * S;
  pc::k_cmac_stream_tma<S><<<grid, dim3(288, 1, 1), smem, h->s_launch>>>(S_);
#endif
  return 0;
}

int launch_cmac_stream_tma(b200conv* h, const pc::CmacParams& P, int C, int stages, int per_sm, bool dynamic = false, float skew = -1.0f) {
  pc::StreamParams S{};
  S.H = P.H; S.h_cstride = P.h_cstride;
  S.X = P.X; S.x_cstride = P.x_cstride; S.xrow0 = P.xrow0;
  S.Y = P.Y; S.y_cstride = P.y_cstride; S.y_rstride = P.y_rstride; S.yrow0 = P.yrow0;
  S.B = P.B; S.P = P.Ppad; S.nblocks = 1;
  const int W = pc::stream_tma_w(P.B), PP = pc::stream_tma_pp(P.B), RG = pc::stream_tma_rg(P.B);
  const int xt = P.B / W;
  // per_sm CTAs per SM, but no CTA with fewer than two ring stages of partitions
  int nsplit = std::max(1, (per_sm * h->n_sm) / std::max(1, xt * C));
  nsplit = std::max(1, std::min(nsplit, std::max(1, P.Ppad / (2 * PP))));
  S.nsplit = nsplit;
  if (!dynamic && (nsplit > 1 || RG > 1))
    CU_CHECK(h, cudaMemsetAsync(S.Y + S.yrow0 * S.y_rstride, 0, (size_t)S.y_rstride * sizeof(float2), h->s_launch));
  dim3 grid(xt, nsplit, C);
  if (!dynamic && h->opt_stream_alt) S.descending = (int)(h->stream_launches++ & 1u);
  if (skew >= 0.0f && !dynamic) {        // skewed static slices, channels interleaved in launch order
    S.interleave = 1; S.skew = skew;
    grid = dim3(xt, nsplit * C, 1);
  }
  if (dynamic) {
    if (xt * C > 256) return fail(h, B200CONV_EINVAL, "too many ticket counters");
    if (!h->stream_ticket) {
      CU_CHECK(h, cudaMalloc(&h->stream_ticket, 256 * sizeof(unsigned long long)));
      CU_CHECK(h, cudaMemsetAsync(h->stream_ticket, 0, 256 * sizeof(unsigned long long), h->s_launch));
      h->stream_ticket_base = 0;
    }
    nsplit = std::max(1, std::min((per_sm * h->n_sm) / std::max(1, xt * C), std::max(1, P.Ppad / (2 * PP))));
    S.nsplit = nsplit;
    grid = dim3(xt, nsplit, C);
    S.ticket = h->stream_ticket; S.ticket_base = h->stream_ticket_base; S.chunk_stages = 2;
    h->stream_ticket_base += (unsigned long long)pc::stream_dyn_chunks(S.P, PP, S.chunk_stages) + (unsigned long long)nsplit;
    CU_CHECK(h, cudaMemsetAsync(S.Y + S.yrow0 * S.y_rstride, 0, (size_t)S.y_rstride * sizeof(float2), h->s_launch));   // always RED.ADD
    int idd = timing_begin(h, kKindCmac);
    if (stages == 12) launch_stream_tma_dyn_s<12>(h, S, grid); else launch_stream_tma_dyn_s<6>(h, S, grid);
    timing_end(h, idd);
    h->launches++;
    CU_CHECK(h, cudaGetLastError());
    return 0;
  }
  int id = timing_begin(h, kKindCmac);
  switch (stages) {
    case 2: launch_stream_tma_s<2>(h, S, grid); break;
    case 6: launch_stream_tma_s<6>(h, S, grid); break;
    case 12: launch_stream_tma_s<12>(h, S, grid); break;
    default: launch_stream_tma_s<4>(h, S, grid); break;
  }
  timing_end(h, id);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

// ---- tensor-core sweep (kernels_tc.cuh) -------------------------------------------------------------------------
constexpr int kTcMinBlocks = 4096;      // below that a 128-segment tile is mostly padding: the FFMA sweep is faster
constexpr int kTfftMinBins = 256;       // automatic FFT sweep along the block axis: the range it was measured in
constexpr int kTfftMinParts = 256;

// can this sweep run on the tensor cores?  (geometry only; the scratch is allocated by launch_cmac_tc)
bool tc_eligible(const b200conv* h, const pc::CmacParams& P, int C) {
#if defined(PC_EMULATE)
  (void)h; (void)P; (void)C;
  return false;
#else
  if (P.xg > 0 || P.Ppad < 1 || P.nblocks < 1) return false;
  const pc::tc::Geom g = pc::tc::make_geom(P.Ppad, P.nblocks);
  if (!pc::tc::geom_ok(g, P.B)) return false;
  return (unsigned long long)C * P.B * 4ull * (unsigned long long)g.rows < (1ull << 31);
#endif
}

// grow-only device scratch; a failed allocation is not an error of the call (the caller falls back to another
// sweep and sets *failed so that later launch groups do not try again)
template <class T>
bool grow_reserve(T** buf, size_t* have, size_t need, bool* failed) {
  if (*have >= need) return true;
  cudaFree(*buf);
  *buf = nullptr; *have = 0;
  if (cudaMalloc((void**)buf, need) != cudaSuccess) { cudaGetLastError(); *buf = nullptr; *failed = true; return false; }
  *have = need;
  return true;
}

// returns 1 when the scratch could not be allocated (nothing launched), 0 on success, < 0 on error
int launch_cmac_tc(b200conv* h, const pc::CmacParams& P, int C) {
#if defined(PC_EMULATE)
  (void)P; (void)C;
  return fail(h, B200CONV_EINVAL, "the tensor-core sweep is not part of the CPU emulation");
#else
  namespace tc = pc::tc;
  const tc::Geom g = tc::make_geom(P.Ppad, P.nblocks);
  const size_t lines = (size_t)C * P.B;
  if (!h->tc_err) {
    CU_CHECK(h, cudaHostAlloc((void**)&h->tc_err, sizeof(int), cudaHostAllocMapped));
    *h->tc_err = 0;
    CU_CHECK(h, cudaHostGetDevicePointer((void**)&h->tc_err_dev, h->tc_err, 0));
  }
  if (*reinterpret_cast<volatile int*>(h->tc_err) != 0)
    return fail(h, B200CONV_ECUDA, "tensor-core sweep: a pipeline barrier timed out (code " + std::to_string(*h->tc_err) + ")");
  if (!grow_reserve(&h->tc_Xt, &h->tc_Xt_bytes, lines * 4 * (size_t)g.Lt * sizeof(float), &h->tc_alloc_failed)) return 1;
  if (!grow_reserve(&h->tc_Yt, &h->tc_Yt_bytes, lines * 4 * (size_t)g.Lty * sizeof(float), &h->tc_alloc_failed)) return 1;
  const size_t a_bytes = lines * (size_t)g.nchunk * 2 * tc::kATileBytes;
  const bool a_stale = h->tc_A_for != P.H || h->tc_A_P != P.Ppad || h->tc_A_B != P.B || h->tc_A_C != C || h->tc_A_bytes < a_bytes;
  if (a_stale) {
    h->tc_A_for = nullptr;
    if (!grow_reserve(&h->tc_A, &h->tc_A_bytes, a_bytes, &h->tc_alloc_failed)) return 1;
  }
  if (!h->tc_attr_set) {
    CU_CHECK(h, cudaFuncSetAttribute(tc::k_tc_sweep, cudaFuncAttributeMaxDynamicSharedMemorySize, tc::kSmemBytes));
    h->tc_attr_set = true;
  }
  cudaStream_t st = h->s_launch;
  int id = timing_begin(h, kKindCmac);
  if (a_stale) {     // once per IR (and stage): H -> tf32 hi / lo Toeplitz tile images
    tc::BuildAParams bp{P.H, P.h_cstride, P.B, P.Ppad, g.Q, g.nchunk, h->tc_A};
    tc::k_tc_build_a<<<dim3(g.nchunk, P.B, C), 256, 0, st>>>(bp);
    h->tc_A_for = P.H; h->tc_A_P = P.Ppad; h->tc_A_B = P.B; h->tc_A_C = C;
    h->launches++;
  }
  tc::SplitXParams sp{P.X, P.x_cstride, P.xrow0 - g.Q, std::max<long long>(0, P.xrow0 - (P.Ppad - 1)), P.xrow0 + P.nblocks, P.B, g.rows, h->tc_Xt};
  tc::k_tc_split_x<<<dim3((unsigned)(g.rows * 2), P.B / 32, C), dim3(32, 8), 0, st>>>(sp);
  tc::SweepParams wp{h->tc_A, h->tc_Xt, h->tc_Yt, (int)lines, g.ntile, g.nchunk, g.rows, g.Lty, 0, h->tc_err_dev};
  const int total = (int)lines * g.ntile;
  tc::k_tc_sweep<<<std::min(total, h->n_sm), tc::kThreads, tc::kSmemBytes, st>>>(wp);
  tc::MergeYParams mp{h->tc_Yt, g.Lty, P.B, P.nblocks, P.Y, P.y_cstride, P.y_rstride, P.yrow0};
  tc::k_tc_merge_y<<<dim3((P.nblocks + 31) / 32, P.B / 32, C), dim3(32, 8), 0, st>>>(mp);
  timing_end(h, id);
  h->launches += 3;
  CU_CHECK(h, cudaGetLastError());
  return 0;
#endif
}

// ---- FFT sweep along the block axis (kernels_tfft.cuh) ---------------------------------------------------------
// cmac_variant 50: N = 4096, G = 4 (the automatic choice); 51: N = 2048, G = 4; 52: N = 2048, G = 8
struct TfftShape { int N, G; };
inline TfftShape tfft_shape(int variant) {
  return variant == 51 ? TfftShape{2048, 4} : variant == 52 ? TfftShape{2048, 8} : TfftShape{4096, 4};
}

bool tfft_eligible(const pc::CmacParams& P, int C, int variant) {
  const TfftShape s = tfft_shape(variant);
  if (P.xg > 0 || P.Ppad < 1 || P.nblocks < 1 || P.B % s.G != 0) return false;
  if (P.Ppad - 1 > pc::tfft_qmax(s.N)) return false;
  const pc::TfftGeom g = pc::tfft_geom(s.N, P.Ppad, P.nblocks);
  return (unsigned long long)C * (P.B / s.G) * (unsigned long long)g.nseg < (1ull << 31);
}

template <int N, int G>
void tfft_launch_t(b200conv* h, const pc::TfftBuildParams* bp, const pc::TfftParams& wp, int C, int ntiles) {
#if defined(PC_EMULATE)
  if (bp) pc::emu_tfft_build_h<N, G>(C, *bp);
  pc::emu_tfft_sweep<N, G>(C, wp);
  (void)h; (void)ntiles;
#else
  constexpr size_t smem = pc::tfft_smem_bytes(N, G);
  constexpr int nt = pc::tfft_threads(N, G);
  if (bp) pc::k_tfft_build_h<N, G><<<dim3(bp->B / G, C), nt, smem, h->s_launch>>>(*bp);
  pc::k_tfft_sweep<N, G><<<ntiles, nt, smem, h->s_launch>>>(wp);
#endif
}

// returns 1 when the filter spectra could not be allocated (nothing launched), 0 on success, < 0 on error
int launch_cmac_tfft(b200conv* h, const pc::CmacParams& P, int C, int variant) {
  const TfftShape s = tfft_shape(variant);
  const size_t hf_bytes = (size_t)C * P.B * s.N * sizeof(float2);
  const bool stale = h->tfft_Hf_for != P.H || h->tfft_Hf_P != P.Ppad || h->tfft_Hf_B != P.B || h->tfft_Hf_C != C ||
                     h->tfft_Hf_N != s.N || h->tfft_Hf_bytes < hf_bytes;
  if (stale) {
    h->tfft_Hf_for = nullptr;
    if (!grow_reserve(&h->tfft_Hf, &h->tfft_Hf_bytes, hf_bytes, &h->tfft_alloc_failed)) return 1;
  }
  if (h->tfft_tw_N != s.N) {
    const std::vector<float2> tw = fft_twiddles(s.N);
    h->tfft_tw_N = 0;
    if (!grow_reserve(&h->tfft_tw, &h->tfft_tw_bytes, tw.size() * sizeof(float2), &h->tfft_alloc_failed)) return 1;
    CU_CHECK(h, cudaMemcpyAsync(h->tfft_tw, tw.data(), tw.size() * sizeof(float2), cudaMemcpyHostToDevice, h->s_launch));
    CU_CHECK(h, cudaStreamSynchronize(h->s_launch));
    h->tfft_tw_N = s.N;
  }
#if !defined(PC_EMULATE)
  const int vi = variant - 50;
  if (!h->tfft_attr_set[vi]) {
    if (variant == 51) {
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_sweep<2048, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(2048, 4)));
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_build_h<2048, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(2048, 4)));
    } else if (variant == 52) {
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_sweep<2048, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(2048, 8)));
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_build_h<2048, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(2048, 8)));
    } else {
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_sweep<4096, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(4096, 4)));
      CU_CHECK(h, cudaFuncSetAttribute(pc::k_tfft_build_h<4096, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)pc::tfft_smem_bytes(4096, 4)));
    }
    h->tfft_attr_set[vi] = true;
  }
#endif
  const pc::TfftGeom g = pc::tfft_geom(s.N, P.Ppad, P.nblocks);
  pc::TfftBuildParams bp{P.H, P.h_cstride, h->tfft_Hf, h->tfft_tw, P.B, P.Ppad};
  pc::TfftParams wp{P.X, P.x_cstride, P.xrow0, std::max<long long>(0, P.xrow0 - (P.Ppad - 1)), P.xrow0 + P.nblocks,
                    h->tfft_Hf, P.Y, P.y_cstride, P.y_rstride, P.yrow0, h->tfft_tw, P.B, P.nblocks, g.Q, g.Lo, g.nseg};
  const int ntiles = C * (P.B / s.G) * g.nseg;
  int id = timing_begin(h, kKindCmac);
  switch (variant) {     // once per IR (and stage) the filter spectra first, then the sweep
    case 51: tfft_launch_t<2048, 4>(h, stale ? &bp : nullptr, wp, C, ntiles); break;
    case 52: tfft_launch_t<2048, 8>(h, stale ? &bp : nullptr, wp, C, ntiles); break;
    default: tfft_launch_t<4096, 4>(h, stale ? &bp : nullptr, wp, C, ntiles); break;
  }
  timing_end(h, id);
  if (stale) {
    h->tfft_Hf_for = P.H; h->tfft_Hf_P = P.Ppad; h->tfft_Hf_B = P.B; h->tfft_Hf_C = C; h->tfft_Hf_N = s.N;
    h->launches++;
  }
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

// P.Ppad enters as the number of real (unpadded) partition rows of this shard
int launch_cmac(b200conv* h, const pc::CmacParams& P, int C) {
  int variant = h->cfg.cmac_variant;
  if (P.xg > 0 && variant >= 50 && variant <= 52)
    return fail(h, B200CONV_EINVAL, "FFT sweep along the block axis: the slot exchange is not supported");
  if (P.xg > 0) variant = (P.nblocks >= 64) ? 22 : 26;     // slot exchange: only the packed-FMA sweeps carry the exchange epilogue
  if (variant == 0) {
    // streaming sweep for real-time calls; packed-FMA batched sweep otherwise (TT = 16 when the
    // launch group is long enough to fill 16-block tiles, TT = 8 below that)
    if (P.nblocks == 1 && P.B >= 64 && P.Ppad >= 1) {
      // TMA ring: 6 stages x 2 CTAs/SM for working sets beyond L2 and multi-tile rows (0.81 of the HBM peak on the
      // 120 s IR, 0.98 on an 8192-bin tail stage); 12 stages x 1 CTA/SM for rows below 512 bins and L2-resident
      // single-tile shapes (fewer CTAs to ramp up) — profiles/r02_stream_variants2.txt
      const size_t bytes = (size_t)P.Ppad * P.B * 16 * (size_t)C;
      variant = (P.B < 512 || (P.B == 512 && bytes <= (size_t)32 << 20)) ? 104 : 103;
    }
    else if (P.nblocks <= kStreamNBS && P.B >= 64 && P.Ppad >= 1) variant = 101;
    else if (P.nblocks <= kStreamNBS && P.B >= 2 && P.Ppad >= 1) variant = 100;
    // FFT along the block axis where it measured faster than the tensor-core sweep (profiles/r03_*)
    else if (h->opt_tfft && !h->tfft_alloc_failed && P.nblocks >= kTcMinBlocks && P.B >= kTfftMinBins &&
             P.Ppad >= kTfftMinParts && tfft_eligible(P, C, 50)) variant = 50;
    else if (h->opt_tc && !h->tc_alloc_failed && P.nblocks >= kTcMinBlocks && tc_eligible(h, P, C)) variant = 40;
    else variant = (P.nblocks >= 64) ? 22 : 26;
  }
  h->last_variant = variant;
  if (variant >= 50 && variant <= 52) {
    if (!tfft_eligible(P, C, variant))
      return fail(h, B200CONV_EINVAL, "FFT sweep along the block axis: unsupported shape (needs B a multiple of the bin group, "
                                      "P - 1 <= 3/4 of the transform length, no slot exchange)");
    const int rc = launch_cmac_tfft(h, P, C, variant);
    if (rc <= 0) return rc;
    if (h->cfg.cmac_variant == variant) return fail(h, B200CONV_ENOMEM, "FFT sweep along the block axis: filter spectra allocation failed");
    // not enough device memory for the spectra
    variant = (h->opt_tc && !h->tc_alloc_failed && P.nblocks >= kTcMinBlocks && tc_eligible(h, P, C)) ? 40 : (P.nblocks >= 64) ? 22 : 26;
    h->last_variant = variant;
  }
  if (variant == 40) {                         // tcgen05 3xTF32 block-Toeplitz sweep
    if (!tc_eligible(h, P, C)) return fail(h, B200CONV_EINVAL, "tensor-core sweep: unsupported shape (needs B % 32 == 0, at most 961 partitions, no slot exchange)");
    const int rc = launch_cmac_tc(h, P, C);
    if (rc <= 0) return rc;
    if (h->cfg.cmac_variant == 40) return fail(h, B200CONV_ENOMEM, "tensor-core sweep: scratch allocation failed");
    variant = (P.nblocks >= 64) ? 22 : 26;     // not enough device memory for the scratch: FFMA sweep
    h->last_variant = variant;
  }
  if (variant == 108) {                        // 6 stages x 2 CTAs/SM, skewed static slices (B200CONV_STREAM_SKEW percent, default 8)
    if (P.nblocks != 1 || P.B < 64) return fail(h, B200CONV_EINVAL, "TMA streaming sweep needs nblocks == 1 and B >= 64");
    static const float skew = [] { const char* e = std::getenv("B200CONV_STREAM_SKEW"); return e ? (float)std::atof(e) / 100.0f : 0.08f; }();
    return launch_cmac_stream_tma(h, P, C, 6, 2, false, skew);
  }
  if (variant == 106 || variant == 107) {      // dynamic chunk tickets: 106 = 6 stages x 2 CTAs/SM, 107 = 12 x 1
    if (P.nblocks != 1 || P.B < 64) return fail(h, B200CONV_EINVAL, "TMA streaming sweep needs nblocks == 1 and B >= 64");
    return launch_cmac_stream_tma(h, P, C, variant == 106 ? 6 : 12, variant == 106 ? 2 : 1, true);
  }
  if (variant >= 102 && variant <= 105) {
    if (P.nblocks != 1 || P.B < 64) return fail(h, B200CONV_EINVAL, "TMA streaming sweep needs nblocks == 1 and B >= 64");
    // 102: 4 stages x 3 CTAs/SM   103: 6 x 2   104: 12 x 1   105: 2 x 6    (all 192 KB in flight per SM)
    static const int cfg[4][2] = {{4, 3}, {6, 2}, {12, 1}, {2, 6}};
    return launch_cmac_stream_tma(h, P, C, cfg[variant - 102][0], cfg[variant - 102][1]);
  }
  if (variant == 101) {
    if (P.nblocks > kStreamNBS || P.B < 4) return fail(h, B200CONV_EINVAL, "streaming sweep needs nblocks <= 4 and B >= 4");
    return launch_cmac_stream_rows(h, P, C);
  }
  if (variant == 100) {
    if (P.nblocks > kStreamNBS || P.B < 2) return fail(h, B200CONV_EINVAL, "streaming sweep needs nblocks <= 4 and B >= 2");
    return launch_cmac_stream(h, P, C);
  }
  int id = timing_begin(h, kKindCmac);
  switch (variant) {
    case 1: launch_cmac_t<16, 4, 8>(h, P, C); break;
    case 2: launch_cmac_t<16, 4, 4>(h, P, C); break;
    case 3: launch_cmac_t<8, 4, 4>(h, P, C); break;
    case 4: launch_cmac_t<8, 4, 8>(h, P, C); break;
    case 5: launch_cmac_t<16, 2, 8>(h, P, C); break;
    case 6: launch_cmac_t<32, 4, 4>(h, P, C); break;
    case 7: launch_cmac_t<4, 4, 8>(h, P, C); break;
    case 11: launch_cmac_bs<16, 4, 8>(h, P, C); break;
    case 12: launch_cmac_bs<16, 4, 4>(h, P, C); break;
    case 16: launch_cmac_bs<32, 4, 4>(h, P, C); break;
    case 21: launch_cmac2_bs<16, 4, 4, 4>(h, P, C); break;    // FFMA2, 128 thr/CTA, <=128 regs
    case 22: launch_cmac2_bs<16, 4, 4, 3>(h, P, C); break;    // FFMA2, 128 thr/CTA, <=168 regs
    case 23: launch_cmac2_bs<16, 4, 8, 2>(h, P, C); break;    // FFMA2, 256 thr/CTA, <=128 regs
    case 24: launch_cmac2_bs<16, 2, 4, 4>(h, P, C); break;
    case 25: launch_cmac2_bs<12, 4, 4, 4>(h, P, C); break;
    case 26: launch_cmac2_bs<8, 4, 4, 4>(h, P, C); break;
    case 27: launch_cmac2_bs<16, 4, 2, 8>(h, P, C); break;    // 64 thr/CTA
    case 28: launch_cmac2_bs<24, 4, 4, 2>(h, P, C); break;
    // banked for the next tuning round (functionally verified, not yet timed):
    case 33: launch_cmac2_bs<16, 8, 4, 3>(h, P, C); break;    // deeper software prefetch
    case 34: launch_cmac2_bs<16, 4, 2, 6>(h, P, C); break;    // 64-thread CTAs, 6 per SM: finer load balance
    default: return fail(h, B200CONV_EINVAL, "unknown cmac_variant");
  }
  timing_end(h, id);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
  return 0;
}

int set_device(b200conv* h) {
  CU_CHECK(h, cudaSetDevice(h->cfg.device));
  return 0;
}

// ---- IR load -------------------------------------------------------------------------------
size_t trimmed_len(const float* ir, size_t n) {
  // FFTConvolver.cpp:103-106 / TwoStageFFTConvolver.cpp:107-110: absolute 1e-6 threshold
  while (n > 0 && std::fabs(ir[n - 1]) < 0.000001f) --n;
  return n;
}

int build_stage(b200conv* h, Stage& s, const float* const* ir, const std::vector<size_t>& L) {
  const int C = h->C;
  const int B = s.B;
  // partitions of this stage (max over channels)
  size_t maxlen = 0;
  std::vector<int> len_c(C, 0);
  for (int c = 0; c < C; ++c) {
    size_t e = std::min(L[c], s.tap_end);
    size_t n = e > s.tap_off ? e - s.tap_off : 0;
    len_c[c] = (int)n;
    maxlen = std::max(maxlen, n);
  }
  s.P_full = (int)((maxlen + B - 1) / B);
  s.q = (int)(s.tap_off / B);
  // shard range
  const int G = std::max(1, h->cfg.shard_count), g = h->cfg.shard_rank;
  const int per = (s.P_full + G - 1) / G;
  s.p_begin = std::min(s.P_full, g * per);
  s.p_end = std::min(s.P_full, (g + 1) * per);
  s.P = s.p_end - s.p_begin;
  s.Prows = round_up(std::max(s.P, 1), kPadP) + kDPre;
  s.hist = s.p_begin + round_up(std::max(s.P, 1), kPadP) + kDPre;

  const std::vector<float2> tw = fft_twiddles(B);
  const int N = (int)tw.size();
  CU_CHECK(h, cudaMalloc(&s.tw, N * sizeof(float2)));
  CU_CHECK(h, cudaMemcpyAsync(s.tw, tw.data(), N * sizeof(float2), cudaMemcpyHostToDevice, h->s_main));
  std::vector<float2> t512;
  if (B == pc::kF512_M) {       // tables of kernels_fft512.cuh, in double
    t512.resize(pc::kF512_TabLen);
    auto w = [](double num, double den) {
      const double a = -2.0 * M_PI * num / den;
      return make_float2((float)std::cos(a), (float)std::sin(a));
    };
    for (int k2 = 0; k2 < 8; ++k2)
      for (int m = 0; m < 64; ++m) t512[pc::kF512_T1 + k2 * 64 + m] = w((double)m * k2, 512.0);
    for (int a = 0; a < 8; ++a)
      for (int b = 0; b < 8; ++b) t512[pc::kF512_T2 + a * 8 + b] = w((double)a * b, 64.0);
    for (int k = 0; k < 512; ++k) t512[pc::kF512_TS + k] = w((double)k, 1024.0);
    CU_CHECK(h, cudaMalloc(&s.tab512, t512.size() * sizeof(float2)));
    CU_CHECK(h, cudaMemcpyAsync(s.tab512, t512.data(), t512.size() * sizeof(float2), cudaMemcpyHostToDevice, h->s_main));
  }
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));

  // H: upload this shard's taps, transform
  const size_t hrow = (size_t)B;
  CU_CHECK(h, cudaMalloc(&s.H, (size_t)C * s.Prows * hrow * sizeof(float2)));
  CU_CHECK(h, cudaMemsetAsync(s.H, 0, (size_t)C * s.Prows * hrow * sizeof(float2), h->s_main));
  if (s.P > 0) {
    const size_t taps_per_c = (size_t)s.P * B;
    std::vector<float> host((size_t)C * taps_per_c, 0.0f);
    std::vector<int> nvalid(C, 0);
    for (int c = 0; c < C; ++c) {
      const long long first = (long long)s.p_begin * B;            // within the stage
      long long n = (long long)len_c[c] - first;
      n = std::max(0LL, std::min(n, (long long)taps_per_c));
      nvalid[c] = (int)n;
      if (n > 0 && !h->ir_on_device) std::memcpy(&host[(size_t)c * taps_per_c], ir[c] + s.tap_off + first, (size_t)n * sizeof(float));
    }
    float* dtaps = nullptr; int* dnv = nullptr;
    CU_CHECK(h, cudaMalloc(&dtaps, host.size() * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&dnv, C * sizeof(int)));
    if (h->ir_on_device) {        // taps shaped on the device: no host round trip
      CU_CHECK(h, cudaMemsetAsync(dtaps, 0, host.size() * sizeof(float), h->s_main));
      for (int c = 0; c < C; ++c)
        if (nvalid[c] > 0)
          CU_CHECK(h, cudaMemcpyAsync(dtaps + (size_t)c * taps_per_c, ir[c] + s.tap_off + (size_t)s.p_begin * B,
                                      (size_t)nvalid[c] * sizeof(float), cudaMemcpyDeviceToDevice, h->s_main));
    } else
    CU_CHECK(h, cudaMemcpyAsync(dtaps, host.data(), host.size() * sizeof(float), cudaMemcpyHostToDevice, h->s_main));
    CU_CHECK(h, cudaMemcpyAsync(dnv, nvalid.data(), C * sizeof(int), cudaMemcpyHostToDevice, h->s_main));
    pc::FwdParams fp{};
    fp.src = dtaps; fp.src_cstride = (long long)taps_per_c;
    fp.nvalid_c = dnv; fp.nvalid = 0;
    fp.dst = s.H; fp.dst_cstride = (long long)s.Prows * B; fp.dst_row0 = 0;
    fp.tw = s.tw; fp.tab512 = s.tab512; fp.M = B; fp.nblocks = s.P;
    int rc = launch_fwd(h, fp, C);
    if (rc) { cudaFree(dtaps); cudaFree(dnv); return rc; }
    CU_CHECK(h, cudaStreamSynchronize(h->s_main));
    cudaFree(dtaps); cudaFree(dnv);
  }
  return 0;
}

int alloc_stage_state(b200conv* h, Stage& s) {
  const int C = h->C, B = s.B;
  s.Tcap = (int)(h->Lmax / B) + 2;
  s.R = 2 * s.hist + s.Tcap + kMaxTT;
  CU_CHECK(h, cudaMalloc(&s.X, (size_t)C * s.R * B * sizeof(float2)));
  for (int i = 0; i < 2; ++i) {
    CU_CHECK(h, cudaMalloc(&s.Y[i], (size_t)(1 + s.Tcap) * C * B * sizeof(float2)));
    CU_CHECK(h, cudaEventCreateWithFlags(&s.ev_sweep[i], cudaEventDisableTiming));
    CU_CHECK(h, cudaEventCreateWithFlags(&s.ev_post[i], cudaEventDisableTiming));
  }
  s.in_stride = (size_t)B + h->Lmax;
  CU_CHECK(h, cudaMalloc(&s.inbuf, (size_t)C * s.in_stride * sizeof(float)));
  if (s.q > 0) {
    s.ring = next_pow2((size_t)(s.q + 2) * B + h->Lmax + B);
    CU_CHECK(h, cudaMalloc(&s.fut, (size_t)C * s.ring * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&s.inbuf_alt, (size_t)C * s.in_stride * sizeof(float)));
    for (int i = 0; i < 2; ++i) CU_CHECK(h, cudaEventCreateWithFlags(&s.ev_job[i], cudaEventDisableTiming));
  }
  return 0;
}

int clear_state(b200conv* h) {
  if (h->s_tail) CU_CHECK(h, cudaStreamSynchronize(h->s_tail));
  CU_CHECK(h, cudaStreamSynchronize(h->s_post));
  for (auto& s : h->stages) {
    const int C = h->C, B = s.B;
    CU_CHECK(h, cudaMemsetAsync(s.X, 0, (size_t)C * s.R * B * sizeof(float2), h->s_main));
    for (int i = 0; i < 2; ++i)
      CU_CHECK(h, cudaMemsetAsync(s.Y[i], 0, (size_t)(1 + s.Tcap) * C * B * sizeof(float2), h->s_main));
    s.ybuf = 0;
    CU_CHECK(h, cudaMemsetAsync(s.inbuf, 0, (size_t)C * s.in_stride * sizeof(float), h->s_main));
    if (s.inbuf_alt) CU_CHECK(h, cudaMemsetAsync(s.inbuf_alt, 0, (size_t)C * s.in_stride * sizeof(float), h->s_main));
    if (s.fut) CU_CHECK(h, cudaMemsetAsync(s.fut, 0, (size_t)C * s.ring * sizeof(float), h->s_main));
    s.job_waited[0] = s.job_waited[1] = true;
    s.njobs = 0;
    s.head = s.hist;
    s.blocks_done = 0;
    s.fill = 0;
  }
  h->abs_pos = 0;
  h->yprev_stale = false;
  if (h->Yx[0]) {
    const Stage& s0 = h->stages[0];
    const size_t row = (size_t)h->C * s0.B;
    for (int i = 0; i < 2; ++i) CU_CHECK(h, cudaMemsetAsync(h->Yx[i], 0, (size_t)h->cfg.shard_count * h->xslot * sizeof(float2), h->s_main));
    CU_CHECK(h, cudaMemsetAsync(h->Hh, 0, (size_t)3 * h->cfg.shard_count * row * sizeof(float2), h->s_main));
    h->hidx = 0;
  }
  return 0;
}

int init_impl(b200conv* h, int n_stages, const size_t* blocks, const size_t* offsets,
              const float* const* ir, const size_t* ir_len) {
  if (int rc = set_device(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  CU_CHECK(h, cudaStreamSynchronize(h->s_post));
  if (h->s_tail) CU_CHECK(h, cudaStreamSynchronize(h->s_tail));
  free_all(h);
  const int C = h->C;
  for (int s = 0; s < n_stages; ++s)
    if (blocks[s] == 0) return fail(h, B200CONV_EINVAL, "block size 0");
  std::vector<size_t> L(C);
  size_t Lir = 0;
  for (int c = 0; c < C; ++c) {
    if (h->ir_on_device) L[c] = (ir && ir[c] && h->ir_trimmed) ? std::min(h->ir_trimmed[c], ir_len[c]) : 0;
    else L[c] = (ir && ir[c] && ir_len) ? trimmed_len(ir[c], ir_len[c]) : 0;
    Lir = std::max(Lir, L[c]);
  }
  h->ir_len = L;
  if (Lir == 0) return B200CONV_OK;      // empty IR: legal, process() writes zeros (FFTConvolver.cpp:108-111)

  std::vector<Stage> st;
  for (int s = 0; s < n_stages; ++s) {
    Stage x;
    // FFTConvolver.cpp:113 rounds up to a power of two.  Partition sizes above 8192 are clamped to 8192: the
    // output of a partitioned convolver is the same linear convolution whatever the partition size, and
    // every offset that is a multiple of a larger power of two is a multiple of 8192 too (REEV-R asks for
    // tail = max(8192, 2*head), StereoConvolver.cpp:15, i.e. 16384 for host blocks above 4096 samples).
    const size_t b = std::min(next_pow2(blocks[s]), size_t(1) << kMaxBlockLog2);
    x.B = (int)b;
    x.tap_off = offsets ? offsets[s] : 0;
    x.tap_end = (s + 1 < n_stages) ? offsets[s + 1] : Lir;
    if (x.tap_off >= Lir) break;                              // IR shorter than this stage's offset
    x.tap_end = std::min(x.tap_end, Lir);
    if (s > 0 && (x.tap_off % b != 0 || x.tap_off < b))
      return fail(h, B200CONV_EINVAL, "stage offset must be a multiple of (and >=) its block size");
    st.push_back(x);
  }
  const int B0 = st[0].B;
  // default launch-group size: 4736 head blocks, but no more than ~4 M samples of staging per channel
  int batch = h->cfg.max_batch_blocks > 0 ? h->cfg.max_batch_blocks
                                          : std::max(64, std::min(kDefaultBatch, (int)((size_t)4194304 / (size_t)B0)));
  h->Lmax = (size_t)batch * B0;
  for (auto& x : st) h->Lmax = std::max(h->Lmax, (size_t)2 * x.B);
  h->stages = st;
  for (auto& s : h->stages) {
    if (int rc = build_stage(h, s, ir, L)) return rc;
    if (int rc = alloc_stage_state(h, s)) return rc;
  }
  for (int i = 0; i < 2; ++i) {
    CU_CHECK(h, cudaMalloc(&h->din[i], (size_t)C * h->Lmax * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&h->dout[i], (size_t)C * h->Lmax * sizeof(float)));
  }
  CU_CHECK(h, cudaMalloc(&h->dch[0], (size_t)C * h->Lmax * sizeof(float)));
  // latency path staging (calls of up to max(64 head blocks, 16384) samples)
  h->hpin_cap = std::min(h->Lmax, std::max((size_t)64 * B0, (size_t)16384));
  CU_CHECK(h, cudaMallocHost((void**)&h->hpin_in, (size_t)C * h->hpin_cap * sizeof(float)));
  CU_CHECK(h, cudaMallocHost((void**)&h->hpin_out, (size_t)C * h->hpin_cap * sizeof(float)));
  CU_CHECK(h, cudaMallocHost((void**)&h->hflag, 64));
  *h->hflag = 0; h->flag_epoch = 0;
#if defined(PC_EMULATE)
  h->hpin_in_dev = h->hpin_in; h->hpin_out_dev = h->hpin_out; h->hflag_dev = h->hflag;
#else
  if (cudaHostGetDevicePointer((void**)&h->hflag_dev, h->hflag, 0) != cudaSuccess) { cudaGetLastError(); h->hflag_dev = nullptr; }
  if (cudaHostGetDevicePointer((void**)&h->hpin_in_dev, h->hpin_in, 0) != cudaSuccess ||
      cudaHostGetDevicePointer((void**)&h->hpin_out_dev, h->hpin_out, 0) != cudaSuccess) {
    cudaGetLastError();
    h->hpin_in_dev = h->hpin_out_dev = nullptr;       // no zero-copy I/O: the real-time path stays on the copy path
  }
#endif
  if (int rc = clear_state(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  return B200CONV_OK;
}

// A failed load (e.g. B200CONV_ENOMEM for an IR that does not fit) leaves the handle in the "no IR" state:
// nothing half-allocated, later init / process calls work.
int init_common(b200conv* h, int n_stages, const size_t* blocks, const size_t* offsets,
                const float* const* ir, const size_t* ir_len) {
  const int rc = init_impl(h, n_stages, blocks, offsets, ir, ir_len);
  if (rc != B200CONV_OK && !h->sticky_cuda_error) {
    const std::string keep = h->err;
    free_all(h);
    h->err = keep;
  }
  return rc;
}

// copies `count` samples of every convolver channel from the caller's device buffer (n_in routed inputs or
// C plain channels) into a C-channel staging buffer
int copy_in(b200conv* h, float* dst, size_t dstride, const float* src, size_t sstride, size_t count) {
  if (count == 0) return 0;
  if (!h->route_on && !h->route_in_only) {
    CU_CHECK(h, cudaMemcpy2DAsync(dst, dstride * sizeof(float), src, sstride * sizeof(float), count * sizeof(float), h->C,
                                  cudaMemcpyDeviceToDevice, h->s_main));
  } else {
    for (int c = 0; c < h->C; ++c)
      CU_CHECK(h, cudaMemcpyAsync(dst + (size_t)c * dstride, src + (size_t)h->in_map[c] * sstride, count * sizeof(float),
                                  cudaMemcpyDeviceToDevice, h->s_main));
  }
  return 0;
}

void set_cmap(const b200conv* h, pc::FwdParams& fp, bool direct) {
  fp.use_cmap = (direct && (h->route_on || h->route_in_only)) ? 1 : 0;
  for (int c = 0; c < 8; ++c) fp.cmap[c] = h->in_map[c];
}

#if !defined(PC_EMULATE)
#define PC_LAUNCH_MIX(mp, grid, st) pc::k_mix<<<grid, 256, 0, st>>>(mp)
#endif

// per-convolver outputs (C channels in `in`) -> n_out mixed outputs
int launch_mix(b200conv* h, const float* in, size_t in_stride, float* out, size_t out_stride, size_t n, cudaStream_t st) {
#if defined(PC_EMULATE)
  (void)st;
  for (int o = 0; o < h->n_out; ++o)
    for (size_t i = 0; i < n; ++i) {
      float acc = 0.0f;
      for (int c = 0; c < h->C; ++c) {
        const float m = h->mix[o * h->C + c];
        if (m != 0.0f) acc = std::fmaf(m, in[(size_t)c * in_stride + i], acc);
      }
      out[(size_t)o * out_stride + i] = acc;
    }
#else
  pc::MixParams mp{};
  mp.in = in; mp.in_stride = (long long)in_stride; mp.out = out; mp.out_stride = (long long)out_stride;
  mp.n = (long long)n; mp.C = h->C; mp.n_out = h->n_out;
  std::memcpy(mp.mix, h->mix, sizeof(mp.mix));
  dim3 grid((unsigned)((n + 255) / 256), h->n_out, 1);
  PC_LAUNCH_MIX(mp, grid, st);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
#endif
  return 0;
}

// ---- one launch group: n <= Lmax samples, device-resident ------------------------------------
int compact_timeline(b200conv* h, Stage& s) {
  const int C = h->C, B = s.B;
  const size_t bytes = (size_t)s.hist * B * sizeof(float2);
  for (int c = 0; c < C; ++c) {
    float2* base = s.X + (size_t)c * s.R * B;
    CU_CHECK(h, cudaMemcpyAsync(base, base + (size_t)(s.head - s.hist) * B, bytes, cudaMemcpyDeviceToDevice, h->s_launch));
  }
  s.head = s.hist;
  return 0;
}


// ---- slot exchange (fused multi-GPU path) ------------------------------------------------------
struct P2PRecord { unsigned long long kind; unsigned long long ptr; unsigned char ipc[64]; };
constexpr int kP2PBuffers = 8;    // Yx[0], Yx[1], Hh, xout[0], xout[1], flags, din[0], din[1]

int p2p_alloc(b200conv* h) {
  if (h->Yx[0]) return 0;
  const Stage& s = h->stages[0];
  const int G = h->cfg.shard_count, C = h->C, B = s.B;
  const size_t row = (size_t)C * B;
  h->xSR = (s.Tcap + G - 1) / G + 2;
  h->xslot = (size_t)h->xSR * row;
  for (int i = 0; i < 2; ++i) {
    CU_CHECK(h, cudaMalloc(&h->Yx[i], (size_t)G * h->xslot * sizeof(float2)));
    CU_CHECK(h, cudaMemsetAsync(h->Yx[i], 0, (size_t)G * h->xslot * sizeof(float2), h->s_main));
    CU_CHECK(h, cudaMalloc(&h->xout[i], (size_t)C * h->Lmax * sizeof(float)));
  }
  CU_CHECK(h, cudaMalloc(&h->Hh, (size_t)3 * G * row * sizeof(float2)));
  CU_CHECK(h, cudaMemsetAsync(h->Hh, 0, (size_t)3 * G * row * sizeof(float2), h->s_main));
  CU_CHECK(h, cudaMalloc(&h->xflags, 32 * sizeof(unsigned int)));
  CU_CHECK(h, cudaMemsetAsync(h->xflags, 0, 32 * sizeof(unsigned int), h->s_main));
  for (int i = 0; i < 2; ++i)
    if (!h->ev_b1[i]) CU_CHECK(h, cudaEventCreateWithFlags(&h->ev_b1[i], cudaEventDisableTiming));
#if !defined(PC_EMULATE)
  // Load every kernel / driver copy routine the exchange flow launches NOW: a lazy module load
  // synchronises the context and must not happen while a peer's flag barrier is spinning on this device.
  {
    cudaFuncAttributes fa;
    CU_CHECK(h, cudaFuncGetAttributes(&fa, pc::k_p2p_barrier));
    CU_CHECK(h, cudaFuncGetAttributes(&fa, pc::k_copy_rows));
#define PC_PRELOAD(BS) \
    CU_CHECK(h, cudaFuncGetAttributes(&fa, pc::k_cmac_batch2<16, 4, 4, BS, 3>)); \
    CU_CHECK(h, cudaFuncGetAttributes(&fa, pc::k_cmac_batch2<8, 4, 4, BS, 4>));
    PC_PRELOAD(0) PC_PRELOAD(128) PC_PRELOAD(512) PC_PRELOAD(8192)
#undef PC_PRELOAD
    // strided device-to-device copies and memsets as used by run_group_p2p / compact_timeline
    CU_CHECK(h, cudaMemcpy2DAsync(h->Yx[1], h->xslot * sizeof(float2), h->Hh, row * sizeof(float2), row * sizeof(float2), G,
                                  cudaMemcpyDeviceToDevice, h->s_main));
    CU_CHECK(h, cudaMemcpy2DAsync(h->xout[1], h->Lmax * sizeof(float), h->xout[0], h->Lmax * sizeof(float), sizeof(float), C,
                                  cudaMemcpyDeviceToDevice, h->s_post));
    CU_CHECK(h, cudaMemcpyAsync(h->Yx[1], h->Yx[0], row * sizeof(float2), cudaMemcpyDeviceToDevice, h->s_main));
    CU_CHECK(h, cudaMemsetAsync(h->Yx[1], 0, (size_t)G * h->xslot * sizeof(float2), h->s_main));
    CU_CHECK(h, cudaStreamSynchronize(h->s_post));
  }
#endif
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  return 0;
}

// after a host synchronisation: did a flag barrier give up waiting for a peer?
int p2p_check(b200conv* h) {
#if !defined(PC_EMULATE)
  if (h->xflags && h->bar_epoch + h->in_epoch > 0) {
    unsigned int err = 0;
    CU_CHECK(h, cudaMemcpy(&err, h->xflags + 8, sizeof(err), cudaMemcpyDeviceToHost));
    if (err != 0) {
      // report once, then re-arm: one slow peer must not fail every later call
      CU_CHECK(h, cudaMemset(h->xflags + 8, 0, sizeof(unsigned int)));
      return fail(h, B200CONV_ECUDA, "slot-exchange barrier timed out waiting for a peer GPU (audio of this call is incomplete)");
    }
  }
#else
  (void)h;
#endif
  return 0;
}

// bank 0: exchange barriers (flag words 0..7, issued on s_post); bank 1: "input landed" barriers (words 16..23)
int p2p_barrier(b200conv* h, cudaStream_t st, int bank = 0) {
  unsigned int& epoch = bank == 0 ? h->bar_epoch : h->in_epoch;
  epoch++;
#if defined(PC_EMULATE)
  (void)st;
  if (!h->host_barrier) return fail(h, B200CONV_ESTATE, "emulated slot exchange needs a host barrier");
  if (h->host_barrier(h->host_barrier_user) != 0) return fail(h, B200CONV_ECUDA, "host barrier failed");
#else
  if (h->host_barrier) {
    // all shards in ONE process on one device (tests): spinning flag kernels of several handles share the
    // device's hardware queues / copy engines and can block each other, so synchronise through the host
    CU_CHECK(h, cudaStreamSynchronize(st));
    if (h->host_barrier(h->host_barrier_user) != 0) return fail(h, B200CONV_ECUDA, "host barrier failed");
    return 0;
  }
  pc::BarrierParams bp{};
  for (int g = 0; g < h->cfg.shard_count; ++g) bp.peer_flags[g] = h->peer_flags[g] + 16 * bank;
  bp.my_flags = h->xflags + 16 * bank;
  bp.error_word = h->xflags + 8;
  bp.rank = h->cfg.shard_rank; bp.G = h->cfg.shard_count; bp.epoch = epoch;
  {
    static const unsigned long long timeout_ms = [] {
      const char* e = std::getenv("B200CONV_P2P_TIMEOUT_MS");
      const long long v = e ? std::atoll(e) : 0;
      return (unsigned long long)(v > 0 ? v : 4000);       // default 4 s (every kernel of the exchange is pre-loaded at attach)
    }();
    bp.timeout_ns = timeout_ms * 1000000ull;
  }
  pc::k_p2p_barrier<<<1, 32, 0, st>>>(bp);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
#endif
  return 0;
}

// device-to-device row copy as a kernel (never a copy-engine copy: see k_copy_rows)
int copy_rows_kernel(b200conv* h, float* dst, size_t dpitch, const float* src, size_t spitch, size_t width, int rows, cudaStream_t st) {
  if (width == 0 || rows == 0) return 0;
#if defined(PC_EMULATE)
  (void)st;
  for (int r = 0; r < rows; ++r) std::memmove(dst + (size_t)r * dpitch, src + (size_t)r * spitch, width * sizeof(float));
#else
  dim3 grid((unsigned)((width + 255) / 256), rows, 1);
  pc::k_copy_rows<<<grid, 256, 0, st>>>(dst, (long long)dpitch, src, (long long)spitch, (long long)width, rows);
  h->launches++;
  CU_CHECK(h, cudaGetLastError());
#endif
  return 0;
}

// one launch group of a single-stage sharded handle through the slot exchange
int run_group_p2p(b200conv* h, const float* in_dev, size_t in_stride, float* out_dev, size_t out_stride, size_t n) {
  const int C = h->C, G = h->cfg.shard_count, g = h->cfg.shard_rank;
  Stage& s = h->stages[0];
  const int B = s.B;
  const size_t row = (size_t)C * B;
  cudaStream_t ps = h->s_post;
  if (n == 0) return 0;
  if (n + B > h->Lmax) return fail(h, B200CONV_ESTATE, "launch group larger than the staging buffers");
  const size_t total = (size_t)s.fill + n;
  const int complete = (int)(total / B);
  const int partial = (int)(total % B);
  const int nb = complete + (partial > 0 ? 1 : 0);
  const bool direct = (s.fill == 0);
  if (!direct)
    CU_CHECK(h, cudaMemcpy2DAsync(s.inbuf + s.fill, s.in_stride * sizeof(float), in_dev, in_stride * sizeof(float),
                                  n * sizeof(float), C, cudaMemcpyDeviceToDevice, h->s_main));
  const int yb = s.ybuf;
  const int per = (nb + G - 1) / G;
  if (s.head + nb + kMaxTT > s.R) { if (int rc = compact_timeline(h, s)) return rc; }
  pc::FwdParams fp{};
  fp.src = direct ? in_dev : s.inbuf;
  fp.src_cstride = direct ? (long long)in_stride : (long long)s.in_stride;
  fp.nvalid_c = nullptr; fp.nvalid = (long long)total;
  fp.dst = s.X; fp.dst_cstride = (long long)s.R * B; fp.dst_row0 = s.head;
  fp.tw = s.tw; fp.tab512 = s.tab512; fp.M = B; fp.nblocks = nb;
  if (int rc = launch_fwd(h, fp, C)) return rc;

  // the exchange buffers of parity yb are free once every GPU finished the inverse FFT of two groups ago
  CU_CHECK(h, cudaStreamWaitEvent(h->s_main, s.ev_post[yb], 0));
  pc::CmacParams cp{};
  cp.H = s.H; cp.h_cstride = (long long)s.Prows * B;
  cp.X = s.X; cp.x_cstride = (long long)s.R * B; cp.xrow0 = s.head - s.p_begin;
  cp.Y = nullptr; cp.y_cstride = B; cp.y_rstride = (long long)row; cp.yrow0 = 0;
  cp.B = B; cp.Ppad = s.P; cp.nblocks = nb;
  cp.xg = G; cp.xrank = g; cp.xper = per; cp.xslot = (long long)h->xslot;
  cp.xhalo_block = complete > 0 ? complete - 1 : -1;
  for (int r = 0; r < G; ++r) cp.xbase[r] = h->peerYx[r][yb];
  cp.xhalo = h->peerHh0 + (size_t)((h->hidx + 1) % 3) * G * row;
  if (int rc = launch_cmac(h, cp, C)) return rc;
  CU_CHECK(h, cudaEventRecord(s.ev_sweep[yb], h->s_main));
  CU_CHECK(h, cudaStreamWaitEvent(ps, s.ev_sweep[yb], 0));

  if (int rc = p2p_barrier(h, ps)) return rc;          // every GPU's partial rows have landed
  CU_CHECK(h, cudaEventRecord(h->ev_b1[h->xgrp & 1], ps));   // ... hence every GPU is done reading this group's input
  h->xgrp++;

  const int j0 = std::min(nb, g * per), j1 = std::min(nb, (g + 1) * per);
  if (j1 > j0) {
    if (g == 0) { // halo of the first slice = last completed row of the previous group (all G partials)
      if (int rc = copy_rows_kernel(h, reinterpret_cast<float*>(h->Yx[yb]), h->xslot * 2,
                                    reinterpret_cast<const float*>(h->Hh + (size_t)h->hidx * G * row), row * 2, row * 2, G, ps)) return rc;
    }
    pc::InvParams ip{};
    ip.Y = h->Yx[yb]; ip.y_cstride = B; ip.y_rstride = (long long)row; ip.yrow0 = 1;
    ip.tw = s.tw; ip.tab512 = s.tab512; ip.M = B; ip.nblocks = j1 - j0; ip.scale = 1.0f / (float)B;
    ip.n_partials = G; ip.partial_stride = (long long)h->xslot;
    ip.dst = h->peer_xout0[yb]; ip.dst_cstride = (long long)h->Lmax;
    ip.index0 = -(long long)s.fill + (long long)j0 * B; ip.lo = 0; ip.hi = (long long)n; ip.mask = -1;
    ip.n_add = 0; ip.abs0 = 0;
    if (int rc = launch_inv(h, ip, C, ps)) return rc;
  }
  if (int rc = p2p_barrier(h, ps)) return rc;          // every slice of the audio is in shard 0's exchange buffer
  if (g == 0 && out_dev) {
    if (int rc = copy_rows_kernel(h, out_dev, out_stride, h->xout[yb], h->Lmax, n, C, ps)) return rc;
  }
  CU_CHECK(h, cudaEventRecord(s.ev_post[yb], ps));

  if (complete > 0) {
    s.ybuf = yb ^ 1;
    h->hidx = (h->hidx + 1) % 3;
    if (partial > 0) {
      const float* tail_src = direct ? in_dev + (size_t)complete * B : s.inbuf + (size_t)complete * B;
      const size_t tail_pitch = direct ? in_stride : s.in_stride;
      CU_CHECK(h, cudaMemcpy2DAsync(s.inbuf, s.in_stride * sizeof(float), tail_src, tail_pitch * sizeof(float),
                                    partial * sizeof(float), C, cudaMemcpyDeviceToDevice, h->s_main));
    }
    s.head += complete;
    s.blocks_done += complete;
  } else if (direct && partial > 0) {
    CU_CHECK(h, cudaMemcpy2DAsync(s.inbuf, s.in_stride * sizeof(float), in_dev, in_stride * sizeof(float),
                                  partial * sizeof(float), C, cudaMemcpyDeviceToDevice, h->s_main));
  }
  s.fill = partial;
  h->abs_pos += (long long)n;
  return 0;
}

int drain_tail(b200conv* h);

// `overlap`: reduce + inverse FFT go to s_post so that they overlap the next group's forward
// FFT + sweep on s_main (double-buffered Y); otherwise everything is issued on s_main.
int run_group(b200conv* h, const float* in_dev, size_t in_stride, float* out_dev, size_t out_stride, size_t n,
              bool overlap) {
  const int C = h->C;
  const bool root = h->cfg.shard_rank == 0;
  if (h->p2p_on) {
    if (h->route_on) return fail(h, B200CONV_ESTATE, "I/O routing is not available on the slot-exchange path");
    return run_group_p2p(h, in_dev, in_stride, out_dev, out_stride, n);
  }
  cudaStream_t ps = overlap ? h->s_post : h->s_main;
  if (n == 0) return 0;
  if (n + h->stages[0].B > h->Lmax) return fail(h, B200CONV_ESTATE, "launch group larger than the staging buffers");
  if (int rc = drain_tail(h)) return rc;
  // stages >= 1 first (their look-ahead output may be consumed by the head within this group)
  for (int si = (int)h->stages.size() - 1; si >= 0; --si) {
    Stage& s = h->stages[si];
    const int B = s.B;
    const size_t row = (size_t)C * B;           // float2 per Y row (all channels)
    const size_t total = (size_t)s.fill + n;
    const int complete = (int)(total / B);
    const int partial = (int)(total % B);
    const int nb = (si == 0) ? complete + (partial > 0 ? 1 : 0) : complete;
    // With an empty open block the forward FFT reads the caller's buffer directly; only a trailing
    // partial block is buffered.  Otherwise the new samples are appended behind the open block's.
    const bool direct = (s.fill == 0);
    if (!direct) { if (int rc = copy_in(h, s.inbuf + s.fill, s.in_stride, in_dev, in_stride, n)) return rc; }
    const int yb = s.ybuf;
    float2* Yb = s.Y[yb];
    if (nb > 0) {
      if (s.head + nb + kMaxTT > s.R) { if (int rc = compact_timeline(h, s)) return rc; }
      pc::FwdParams fp{};
      fp.src = direct ? in_dev : s.inbuf;
      fp.src_cstride = direct ? (long long)in_stride : (long long)s.in_stride;
      fp.nvalid_c = nullptr; fp.nvalid = (long long)total;
      set_cmap(h, fp, direct);
      fp.dst = s.X; fp.dst_cstride = (long long)s.R * B; fp.dst_row0 = s.head;
      fp.tw = s.tw; fp.tab512 = s.tab512; fp.M = B; fp.nblocks = nb;
      if (int rc = launch_fwd(h, fp, C)) return rc;

      // Y[yb] rows >= 1 may still be read by the post work of two groups ago
      if (overlap) CU_CHECK(h, cudaStreamWaitEvent(h->s_main, s.ev_post[yb], 0));
      // overlap state after a forward-FFT-only advance (time-slice sharding): Y row 0 must become
      // sum_p H[p] X[head-1-p], the spectrum of the block in front of this group — its input spectra are in the
      // timeline, so the sweep simply starts one block early and writes that block as row 0
      const int extra = (si == 0 && h->yprev_stale) ? 1 : 0;
      if (extra) {
        if (overlap) CU_CHECK(h, cudaStreamWaitEvent(h->s_main, s.ev_post[yb ^ 1], 0));   // row 0 was written on s_post
        h->yprev_stale = false;
      }
      pc::CmacParams cp{};
      cp.H = s.H; cp.h_cstride = (long long)s.Prows * B;
      cp.X = s.X; cp.x_cstride = (long long)s.R * B; cp.xrow0 = s.head - s.p_begin - extra;
      cp.Y = Yb; cp.y_cstride = B; cp.y_rstride = (long long)row; cp.yrow0 = 1 - extra;
      cp.B = B; cp.Ppad = s.P; cp.nblocks = nb + extra;
      if (int rc = launch_cmac(h, cp, C)) return rc;
      if (overlap) {
        CU_CHECK(h, cudaEventRecord(s.ev_sweep[yb], h->s_main));
        CU_CHECK(h, cudaStreamWaitEvent(ps, s.ev_sweep[yb], 0));
      }

      if (h->cfg.shard_count > 1) {
        if (!h->reduce) return fail(h, B200CONV_ESTATE, "sharded handle without a reduce hook");
        if (h->reduce(h->reduce_user, reinterpret_cast<float*>(Yb + row), (size_t)nb * row * 2, ps) != 0)
          return fail(h, B200CONV_ECUDA, "reduce hook failed");
      }
      if (root) {
        pc::InvParams ip{};
        ip.Y = Yb; ip.y_cstride = B; ip.y_rstride = (long long)row; ip.yrow0 = 1;
        ip.tw = s.tw; ip.tab512 = s.tab512; ip.M = B; ip.nblocks = nb; ip.scale = 1.0f / (float)B;
        if (si == 0) {
          ip.dst = h->route_on ? h->dch[0] : out_dev;
          ip.dst_cstride = h->route_on ? (long long)h->Lmax : (long long)out_stride;
          ip.index0 = -(long long)s.fill; ip.lo = 0; ip.hi = (long long)n; ip.mask = -1;
          ip.abs0 = h->abs_pos - s.fill;
          int na = 0;
          for (size_t sj = 1; sj < h->stages.size() && na < 3; ++sj) {
            ip.add[na] = h->stages[sj].fut; ip.add_cstride[na] = (long long)h->stages[sj].ring;
            ip.add_mask[na] = (long long)h->stages[sj].ring - 1;
            ++na;
          }
          ip.n_add = na;
        } else {
          ip.dst = s.fut; ip.dst_cstride = (long long)s.ring;
          ip.index0 = (s.blocks_done + s.q) * (long long)B;
          ip.lo = 0; ip.hi = (long long)1 << 62; ip.mask = (long long)s.ring - 1;
          ip.n_add = 0; ip.abs0 = 0;
        }
        if (int rc = launch_inv(h, ip, C, ps)) return rc;
        if (si == 0 && h->route_on) { if (int rc = launch_mix(h, h->dch[0], h->Lmax, out_dev, out_stride, n, ps)) return rc; }
      }
    }
    // state update
    if (complete > 0) {
      // overlap state for the next group: last completed row -> row 0 of the buffer it will use
      const int nxt = overlap ? (yb ^ 1) : yb;
      CU_CHECK(h, cudaMemcpyAsync(s.Y[nxt], Yb + (size_t)complete * row, row * sizeof(float2),
                                  cudaMemcpyDeviceToDevice, ps));
      if (overlap) CU_CHECK(h, cudaEventRecord(s.ev_post[yb], ps));
      s.ybuf = nxt;
      if (partial > 0) {
        if (direct) { if (int rc = copy_in(h, s.inbuf, s.in_stride, in_dev + (size_t)complete * B, in_stride, partial)) return rc; }
        else
          CU_CHECK(h, cudaMemcpy2DAsync(s.inbuf, s.in_stride * sizeof(float), s.inbuf + (size_t)complete * B,
                                        s.in_stride * sizeof(float), partial * sizeof(float), C, cudaMemcpyDeviceToDevice, h->s_main));
      }
      s.head += complete;
      s.blocks_done += complete;
    } else {
      if (direct && partial > 0) {   // nothing completed: keep the partial block's samples for the next call
        if (int rc = copy_in(h, s.inbuf, s.in_stride, in_dev, in_stride, partial)) return rc;
      }
      if (overlap && nb > 0) CU_CHECK(h, cudaEventRecord(s.ev_post[yb], ps));
    }
    s.fill = partial;
  }
  h->abs_pos += (long long)n;
  return 0;
}

// Forward FFTs only (uniform handle, no open block): the spectra of `nblocks` input blocks go into the timeline,
// no sweep, no output.  Used by the time-slice sharding for the history in front of a slice and for the tail of
// the call every GPU keeps.
int advance_fft_only(b200conv* h, const float* in_dev, size_t in_stride, long long nblocks) {
  Stage& s = h->stages[0];
  const int C = h->C, B = s.B;
  for (long long done = 0; done < nblocks;) {
    const int nb = (int)std::min<long long>(nblocks - done, s.Tcap);
    if (s.head + nb + kMaxTT > s.R) { if (int rc = compact_timeline(h, s)) return rc; }
    pc::FwdParams fp{};
    fp.src = in_dev + (size_t)done * B; fp.src_cstride = (long long)in_stride;
    fp.nvalid_c = nullptr; fp.nvalid = (long long)nb * B;
    set_cmap(h, fp, false);
    fp.dst = s.X; fp.dst_cstride = (long long)s.R * B; fp.dst_row0 = s.head;
    fp.tw = s.tw; fp.tab512 = s.tab512; fp.M = B; fp.nblocks = nb;
    if (int rc = launch_fwd(h, fp, C)) return rc;
    s.head += nb;
    s.blocks_done += nb;
    done += nb;
  }
  if (nblocks > 0) h->yprev_stale = true;
  h->abs_pos += nblocks * B;
  return 0;
}

// Time-slice sharding of one block-aligned call of T blocks (see b200conv_process_sliced): which blocks this
// GPU transforms only ([lo, a) in front of its slice, [tail_lo, T) behind it) and which it convolves ([a, b)).
struct SlicePlan { long long T, a, b, lo, tail_lo; };

int plan_slice(b200conv* h, size_t len, int rank, int count, SlicePlan* sp) {
  if (count < 1 || rank < 0 || rank >= count) return fail(h, B200CONV_EINVAL, "slice_rank / slice_count out of range");
  if (h->stages.size() != 1) return fail(h, B200CONV_ESTATE, "time-slice sharding needs a uniform (single-stage) handle");
  if (h->cfg.shard_count != 1) return fail(h, B200CONV_ESTATE, "time-slice sharding needs an unsharded handle (the full IR on every GPU)");
  if (h->route_on) return fail(h, B200CONV_ESTATE, "time-slice sharding is not available with I/O routing");
  const Stage& s = h->stages[0];
  if (s.fill != 0 || len % (size_t)s.B != 0)
    return fail(h, B200CONV_ESTATE, "time-slice sharding needs block-aligned calls (len a multiple of the block size, no open block)");
  const long long T = (long long)(len / (size_t)s.B), P = s.P_full;
  const long long per = (T + count - 1) / count;
  sp->T = T;
  sp->a = std::min(T, rank * per);
  sp->b = std::min(T, (rank + 1) * per);
  // block t needs X[t-p], p < P, and the overlap-add needs the spectrum of block t-1 as well: P blocks of history
  sp->lo = sp->b > sp->a ? std::max(0LL, sp->a - P) : sp->a;
  sp->tail_lo = std::max(sp->b, T - P);
  // Without the tail the handle's history ends with its own slice: enough for a following sliced call whose slice
  // starts at least P blocks into the call (it uploads its own history then) — what every rank but 0 of a steady
  // batch job needs; saves P blocks of H2D + forward FFT per call.
  if (!h->opt_slice_tail && sp->b > sp->a) sp->tail_lo = T;
  if (sp->b <= sp->a) { sp->a = sp->b = sp->lo = std::max(0LL, T - P); sp->tail_lo = sp->a; }   // empty slice: only keep the tail
  return 0;
}

// ---- real-time path: one cluster kernel per call (kernels_rt.cuh) + tail blocks on the low-priority stream -----
// every batch-path entry point first orders s_main (and s_post) behind all tail blocks still in flight on s_tail
int drain_tail(b200conv* h) {
  for (auto& s : h->stages)
    for (int j = 0; j < 2; ++j)
      if (!s.job_waited[j]) {
        CU_CHECK(h, cudaStreamWaitEvent(h->s_main, s.ev_job[j], 0));
        CU_CHECK(h, cudaStreamWaitEvent(h->s_post, s.ev_job[j], 0));
        s.job_waited[j] = true;
      }
  return 0;
}

// ONE completed block of a stage >= 1 (its samples are in s.inbuf), everything on h->s_launch: forward FFT into the
// timeline, streaming sweep, inverse FFT into the stage's look-ahead ring (TwoStageFFTConvolver.cpp:201-222)
int run_tail_block(b200conv* h, Stage& s) {
  const int C = h->C, B = s.B;
  const size_t row = (size_t)C * B;
  cudaStream_t st = h->s_launch;
  if (s.head + 1 + kMaxTT > s.R) { if (int rc = compact_timeline(h, s)) return rc; }
  pc::FwdParams fp{};
  fp.src = s.inbuf; fp.src_cstride = (long long)s.in_stride;
  fp.nvalid_c = nullptr; fp.nvalid = (long long)B;
  fp.dst = s.X; fp.dst_cstride = (long long)s.R * B; fp.dst_row0 = s.head;
  fp.tw = s.tw; fp.tab512 = s.tab512; fp.M = B; fp.nblocks = 1;
  if (int rc = launch_fwd(h, fp, C)) return rc;
  float2* Yb = s.Y[s.ybuf];
  pc::CmacParams cp{};
  cp.H = s.H; cp.h_cstride = (long long)s.Prows * B;
  cp.X = s.X; cp.x_cstride = (long long)s.R * B; cp.xrow0 = s.head - s.p_begin;
  cp.Y = Yb; cp.y_cstride = B; cp.y_rstride = (long long)row; cp.yrow0 = 1;
  cp.B = B; cp.Ppad = s.P; cp.nblocks = 1;
  if (int rc = launch_cmac(h, cp, C)) return rc;
  pc::InvParams ip{};
  ip.Y = Yb; ip.y_cstride = B; ip.y_rstride = (long long)row; ip.yrow0 = 1;
  ip.tw = s.tw; ip.tab512 = s.tab512; ip.M = B; ip.nblocks = 1; ip.scale = 1.0f / (float)B;
  ip.dst = s.fut; ip.dst_cstride = (long long)s.ring;
  ip.index0 = (s.blocks_done + s.q) * (long long)B;
  ip.lo = 0; ip.hi = (long long)1 << 62; ip.mask = (long long)s.ring - 1;
  ip.n_add = 0; ip.abs0 = 0;
  if (int rc = launch_inv(h, ip, C, st)) return rc;
  CU_CHECK(h, cudaMemcpyAsync(Yb, Yb + row, row * sizeof(float2), cudaMemcpyDeviceToDevice, st));   // overlap state
  s.head += 1;
  s.blocks_done += 1;
  s.fill = 0;
  return 0;
}

constexpr size_t kRtMaxBytesPerCta = 384 * 1024;      // H + FDL bytes one CTA of the cluster may have to stream

// CTAs per convolver for the cluster kernel; -1 = split mode (head stage too large for one cluster); 0 = the call does not qualify
int rt_cluster_ctas(const b200conv* h, size_t len) {
  if (!h->opt_rt || h->stages.empty() || h->stages.size() > 4) return 0;
  if (h->cfg.shard_count != 1 || h->p2p_on || h->timing || h->yprev_stale) return 0;
  const Stage& s0 = h->stages[0];
  const int M = s0.B, C = h->C;
  if (M < 16 || M > 1024 || C > 8 || len == 0 || (size_t)s0.fill + len > (size_t)M) return 0;
  if (h->route_on && (h->n_out * (int)len > 8 * 1024)) return 0;
  int max_nc = 1;
  while (max_nc * 2 * C <= 16 && max_nc * 2 <= M / 32) max_nc *= 2;     // cluster <= 16 CTAs, tile >= 16 bin pairs
  int nc = 1;
  while (M / nc / 2 > 256) nc *= 2;                                      // at most 256 bin pairs per CTA
  const size_t bytes = (size_t)s0.P * M * 16;                            // H + FDL rows of one convolver
  // one SM pulls ~20-50 GB/s out of L2 with this access pattern: spread a convolver over as many CTAs as the
  // cluster allows until a CTA streams <= 64 KB; beyond kRtMaxBytesPerCta the all-SM streaming sweep wins
  while (nc < max_nc && bytes / nc > 64 * 1024) nc *= 2;
  if (nc > max_nc || bytes / nc > kRtMaxBytesPerCta)
    return (C <= 8 && M >= 64) ? -1 : 0;        // -1: split mode (front kernel, all-SM TMA sweep, back kernel)
  return nc;
}

#if !defined(PC_EMULATE)
template <int M>
cudaError_t rt_launch_m(const pc::RtParams& P, int nctas, size_t smem, cudaStream_t st) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(nctas, 1, 1);
  cfg.blockDim = dim3(256, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute at[1];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = nctas; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, pc::k_rt_block<M>, P);
}
template <int M>
bool rt_set_attr() {
  const int smem = pc::rt_smem_layout(M, 16).bytes;
  return cudaFuncSetAttribute(pc::k_rt_block<M>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem) == cudaSuccess &&
         cudaFuncSetAttribute(pc::k_rt_block<M>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
}
#endif

// One real-time call (rt_cluster_ctas() > 0): `in` / `out` are device-accessible (pinned host or device memory).
int rt_call(b200conv* h, int nc, const float* in, size_t in_stride, float* out, size_t out_stride, size_t len, bool use_flag) {
  const int C = h->C;
  Stage& s0 = h->stages[0];
  const int M = s0.B;
  // tail blocks whose output this call needs must have landed in their look-ahead rings
  for (size_t si = 1; si < h->stages.size(); ++si) {
    Stage& s = h->stages[si];
    for (int j = 0; j < 2; ++j)
      if (!s.job_waited[j] && h->abs_pos + (long long)len > s.job_out_start[j]) {
        CU_CHECK(h, cudaStreamWaitEvent(h->s_main, s.ev_job[j], 0));
        s.job_waited[j] = true;
      }
  }
  if (s0.head + 1 + kMaxTT > s0.R) { if (int rc = compact_timeline(h, s0)) return rc; }
  pc::RtParams P{};
  P.M = M; P.C = C; P.NC = nc; P.P = s0.P;
  P.fill = s0.fill; P.len = (int)len; P.complete = (s0.fill + (int)len == M) ? 1 : 0;
  P.in = in; P.in_stride = (long long)in_stride;
  for (int c = 0; c < 8; ++c) P.in_map[c] = (h->route_on || h->route_in_only) ? h->in_map[c] : c;
  P.inbuf0 = s0.inbuf; P.inbuf0_stride = (long long)s0.in_stride;
  P.H = s0.H; P.h_cstride = (long long)s0.Prows * M;
  P.X = s0.X; P.x_cstride = (long long)s0.R * M; P.head = s0.head;
  P.Yprev = s0.Y[s0.ybuf]; P.Ynext = s0.Y[s0.ybuf ^ 1]; P.y_cstride = M;
  P.tw = s0.tw;
  int na = 0;
  for (size_t si = 1; si < h->stages.size(); ++si) {
    Stage& s = h->stages[si];
    P.later_inbuf[na] = s.inbuf; P.later_stride[na] = (long long)s.in_stride; P.later_fill[na] = s.fill;
    P.add[na] = s.fut; P.add_cstride[na] = (long long)s.ring; P.add_mask[na] = (long long)s.ring - 1;
    ++na;
  }
  P.n_later = na; P.n_add = na;
  P.abs0 = h->abs_pos - s0.fill;
  P.out = out; P.out_stride = (long long)out_stride;
  P.mix_on = h->route_on ? 1 : 0; P.n_out = h->route_on ? h->n_out : C;
  std::memcpy(P.mix, h->mix, sizeof(P.mix));
  const bool split = nc < 0;
  if (split) nc = 1;
  P.NC = nc;
  auto launch = [&](const pc::RtParams& Q) -> int {
#if defined(PC_EMULATE)
    pc::emu_rt_block(Q);
#else
    const size_t smem = (size_t)pc::rt_smem_layout(M, C).bytes;
    cudaError_t e = cudaErrorInvalidValue;
    switch (M) {
      case 16: e = rt_launch_m<16>(Q, C * nc, smem, h->s_main); break;
      case 32: e = rt_launch_m<32>(Q, C * nc, smem, h->s_main); break;
      case 64: e = rt_launch_m<64>(Q, C * nc, smem, h->s_main); break;
      case 128: e = rt_launch_m<128>(Q, C * nc, smem, h->s_main); break;
      case 256: e = rt_launch_m<256>(Q, C * nc, smem, h->s_main); break;
      case 512: e = rt_launch_m<512>(Q, C * nc, smem, h->s_main); break;
      case 1024: e = rt_launch_m<1024>(Q, C * nc, smem, h->s_main); break;
      default: break;
    }
    CU_CHECK(h, e);
#endif
    h->launches++;
    return 0;
  };
  if (!split) {
    if (use_flag && h->hflag_dev) { P.done_flag = h->hflag_dev; P.done_val = ++h->flag_epoch; }
    if (int rc = launch(P)) return rc;
  } else {
    // head stage too large for one cluster: FRONT (assemble + forward FFT + timeline row), the TMA streaming sweep
    // over all SMs into Y row 1, BACK (overlap-add + inverse FFT + output) — still zero-copy I/O and no D2H/H2D
    float2* Yb = s0.Y[s0.ybuf];
    const size_t row = (size_t)C * M;
    P.mode = 1;
    if (int rc = launch(P)) return rc;
    pc::CmacParams cp{};
    cp.H = s0.H; cp.h_cstride = (long long)s0.Prows * M;
    cp.X = s0.X; cp.x_cstride = (long long)s0.R * M; cp.xrow0 = s0.head - s0.p_begin;
    cp.Y = Yb; cp.y_cstride = M; cp.y_rstride = (long long)row; cp.yrow0 = 1;
    cp.B = M; cp.Ppad = s0.P; cp.nblocks = 1;
    if (int rc = launch_cmac(h, cp, C)) return rc;
    P.mode = 2; P.Yt = Yb + row;
    if (use_flag && h->hflag_dev) { P.done_flag = h->hflag_dev; P.done_val = ++h->flag_epoch; }
    if (int rc = launch(P)) return rc;
  }
  // bookkeeping of the head stage
  if (P.complete) { s0.head += 1; s0.blocks_done += 1; s0.fill = 0; s0.ybuf ^= 1; }
  else s0.fill += (int)len;
  h->abs_pos += (long long)len;
  // later stages: the kernel appended the samples; a completed block goes to the low-priority stream
  bool recorded = false;
  for (size_t si = 1; si < h->stages.size(); ++si) {
    Stage& s = h->stages[si];
    s.fill += (int)len;
    if (s.fill < s.B) continue;
    if (!recorded) { CU_CHECK(h, cudaEventRecord(h->ev_rt, h->s_main)); recorded = true; }
    CU_CHECK(h, cudaStreamWaitEvent(h->s_tail, h->ev_rt, 0));
    const int j = (int)(s.njobs & 1);
    s.job_out_start[j] = (s.blocks_done + s.q) * (long long)s.B;
    h->s_launch = h->s_tail;
    const int rc = run_tail_block(h, s);
    h->s_launch = h->s_main;
    if (rc) return rc;
    CU_CHECK(h, cudaEventRecord(s.ev_job[j], h->s_tail));
    s.job_waited[j] = false;
    s.njobs++;
    std::swap(s.inbuf, s.inbuf_alt);              // the following calls fill the other buffer
  }
  return 0;
}

// make s_main wait for everything queued on s_post (end of an overlapped call)
int join_post(b200conv* h) {
  CU_CHECK(h, cudaEventRecord(h->ev_join, h->s_post));
  CU_CHECK(h, cudaStreamWaitEvent(h->s_main, h->ev_join, 0));
  return 0;
}

}  // namespace

// =============================================================================================
// C ABI
// =============================================================================================
extern "C" {

const char* b200conv_version(void) {
#if defined(PC_EMULATE)
  return "b200conv 0.1 EMULATED-ON-CPU (tests only)";
#else
  return "b200conv 0.1 (sm_100a, hand-written Stockham FFT + register-tiled FDL sweep)";
#endif
}

b200conv_t* b200conv_create(const b200conv_config* cfg) {
  if (!cfg || cfg->n_channels < 1) return nullptr;
  b200conv* h = new (std::nothrow) b200conv();
  if (!h) return nullptr;
  h->cfg = *cfg;
  if (h->cfg.shard_count < 1) h->cfg.shard_count = 1;
  if (h->cfg.shard_rank < 0 || h->cfg.shard_rank >= h->cfg.shard_count) h->cfg.shard_rank = 0;
  h->C = cfg->n_channels;
  h->ir_len.assign(h->C, 0);
  // CUDA resources; failures are recorded and reported by the first real call
  if (cudaSetDevice(h->cfg.device) != cudaSuccess) {
    h->err = "cudaSetDevice failed: no usable CUDA device";
    h->sticky_cuda_error = true;
    cudaGetLastError();
    return h;
  }
  int lo = 0, hi = 0;
  cudaDeviceGetStreamPriorityRange(&lo, &hi);
#if !defined(PC_EMULATE)
  {
    int sm = 0;
    if (cudaDeviceGetAttribute(&sm, cudaDevAttrMultiProcessorCount, h->cfg.device) == cudaSuccess && sm > 0) h->n_sm = sm;
  }
#endif
  bool ok = cudaStreamCreateWithPriority(&h->s_main, cudaStreamNonBlocking, hi) == cudaSuccess;
  ok = ok && cudaStreamCreateWithPriority(&h->s_post, cudaStreamNonBlocking, hi) == cudaSuccess;
  // tail blocks have a whole tail period (8192 samples = 171 ms at 48 kHz) to finish: lowest priority, so that they
  // never delay the head-stage kernels of this or any other handle (TwoStageFFTConvolver.cpp:213-222, Convolver.cpp:84-95)
  ok = ok && cudaStreamCreateWithPriority(&h->s_tail, cudaStreamNonBlocking, lo) == cudaSuccess;
  ok = ok && cudaEventCreateWithFlags(&h->ev_rt, cudaEventDisableTiming) == cudaSuccess;
  h->s_launch = h->s_main;
  ok = ok && cudaEventCreateWithFlags(&h->ev_join, cudaEventDisableTiming) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&h->s_in, cudaStreamNonBlocking) == cudaSuccess;
  ok = ok && cudaStreamCreateWithFlags(&h->s_out, cudaStreamNonBlocking) == cudaSuccess;
  for (int i = 0; i < 2 && ok; ++i) {
    ok = ok && cudaEventCreateWithFlags(&h->ev_h2d[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_comp[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_d2h[i], cudaEventDisableTiming) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&h->ev_din[i], cudaEventDisableTiming) == cudaSuccess;
  }
#if !defined(PC_EMULATE)
  if (ok) {
    // function attributes are per device: set them once per device ordinal
    static std::once_flag once[64];
    static bool attr_ok = true;
    std::call_once(once[h->cfg.device & 63], [] {
#define PC_CASE(L) attr_ok = attr_ok && fft_set_smem_attr<L>();
      PC_FOR_EACH_LOG2(PC_CASE)
#undef PC_CASE
      attr_ok = attr_ok && stream_set_smem_attr();
      attr_ok = attr_ok && rt_set_attr<16>() && rt_set_attr<32>() && rt_set_attr<64>() && rt_set_attr<128>() &&
                rt_set_attr<256>() && rt_set_attr<512>() && rt_set_attr<1024>();
      attr_ok = attr_ok && cudaFuncSetAttribute(pc::k_fwd_fft512, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kF512Smem) == cudaSuccess;
      attr_ok = attr_ok && cudaFuncSetAttribute(pc::k_inv_fft512<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kF512Smem) == cudaSuccess;
      attr_ok = attr_ok && cudaFuncSetAttribute(pc::k_inv_fft512<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kF512Smem) == cudaSuccess;
    });
    ok = attr_ok;
  }
#endif
  if (!ok) {
    h->err = std::string("CUDA resource creation failed: ") + cudaGetErrorString(cudaGetLastError());
    h->sticky_cuda_error = true;
  }
  return h;
}

void b200conv_destroy(b200conv_t* h) {
  if (!h) return;
  if (!h->sticky_cuda_error || h->s_main) {
    cudaSetDevice(h->cfg.device);
    if (h->s_main) cudaStreamSynchronize(h->s_main);
    if (h->s_post) cudaStreamSynchronize(h->s_post);
    if (h->s_tail) cudaStreamSynchronize(h->s_tail);
    free_all(h);
    if (h->ev_rt) cudaEventDestroy(h->ev_rt);
    cudaFree(h->stream_ticket); h->stream_ticket = nullptr;
    if (h->s_tail) cudaStreamDestroy(h->s_tail);
    for (auto& p : h->ev_pool) { cudaEventDestroy(p.a); cudaEventDestroy(p.b); }
    for (int i = 0; i < 2; ++i) {
      if (h->ev_h2d[i]) cudaEventDestroy(h->ev_h2d[i]);
      if (h->ev_comp[i]) cudaEventDestroy(h->ev_comp[i]);
      if (h->ev_d2h[i]) cudaEventDestroy(h->ev_d2h[i]);
      if (h->ev_din[i]) cudaEventDestroy(h->ev_din[i]);
    }
    if (h->ev_join) cudaEventDestroy(h->ev_join);
    if (h->s_post) cudaStreamDestroy(h->s_post);
    if (h->s_main) cudaStreamDestroy(h->s_main);
    if (h->s_in) cudaStreamDestroy(h->s_in);
    if (h->s_out) cudaStreamDestroy(h->s_out);
  }
  delete h;
}

const char* b200conv_last_error(const b200conv_t* h) { return h ? h->err.c_str() : "null handle"; }

#define REQUIRE_CUDA(h)                                                   \
  do {                                                                    \
    if (!(h)) return B200CONV_EINVAL;                                     \
    if ((h)->sticky_cuda_error) return B200CONV_ECUDA;                    \
  } while (0)

int b200conv_init_uniform(b200conv_t* h, size_t block, const float* const* ir, const size_t* ir_len) {
  REQUIRE_CUDA(h);
  const size_t off = 0;
  return init_common(h, 1, &block, &off, ir, ir_len);
}

int b200conv_init_twostage(b200conv_t* h, size_t head_block, size_t tail_block,
                           const float* const* ir, const size_t* ir_len) {
  REQUIRE_CUDA(h);
  if (head_block == 0 || tail_block == 0) {                       // TwoStageFFTConvolver.cpp:94-97
    if (int rc = set_device(h)) return rc;
    cudaStreamSynchronize(h->s_main);
    free_all(h);
    return fail(h, B200CONV_EINVAL, "block size 0");
  }
  if (head_block > tail_block) std::swap(head_block, tail_block);  // :100-104
  const size_t hb = next_pow2(head_block), tb = next_pow2(tail_block);   // :117-118
  // head covers taps [0, T), tail0 (same block size as the head, :123-129) taps [T, 2T): the two
  // are one uniform stage of block hb over [0, 2T); the tail runs block T over [2T, L) (:131-138).
  const size_t blocks[2] = {hb, tb};
  const size_t offsets[2] = {0, 2 * tb};
  return init_common(h, 2, blocks, offsets, ir, ir_len);
}

int b200conv_init_stages(b200conv_t* h, int n_stages, const size_t* blocks, const size_t* offsets,
                         const float* const* ir, const size_t* ir_len) {
  REQUIRE_CUDA(h);
  if (n_stages < 1 || n_stages > 4 || !blocks || !offsets || offsets[0] != 0)
    return fail(h, B200CONV_EINVAL, "need 1..4 stages with offsets[0] == 0");
  return init_common(h, n_stages, blocks, offsets, ir, ir_len);
}

// irshape.cu (internal): shape raw host taps into device buffers
int pc_ir_shape_to_device(int device, const float* const* raw, int C, size_t n, const b200conv_ir_shape_params* sp,
                          float** dev_out, size_t* out_len, size_t* trimmed);
void pc_ir_shape_free(float** dev_out, int C);

static int init_shaped(b200conv_t* h, int n_stages, const size_t* blocks, const size_t* offsets,
                       const float* const* raw, size_t n, const b200conv_ir_shape_params* sp) {
  if (!raw || !sp) return fail(h, B200CONV_EINVAL, "null argument");
  if (h->C < 2 || h->C > 8) return fail(h, B200CONV_ESTATE, "IR shaping works on 2..8 channel handles (LL, RR[, LR, RL])");
  float* dev[8] = {};
  size_t m = 0, trimmed[8] = {}, lens[8] = {};
  if (int rc = pc_ir_shape_to_device(h->cfg.device, raw, h->C, n, sp, dev, &m, trimmed))
    return fail(h, rc, "IR shaping on the device failed");
  for (int c = 0; c < h->C; ++c) lens[c] = m;
  h->ir_on_device = true; h->ir_trimmed = trimmed;
  const int rc = init_common(h, n_stages, blocks, offsets, dev, lens);
  h->ir_on_device = false; h->ir_trimmed = nullptr;
  pc_ir_shape_free(dev, h->C);
  return rc;
}

int b200conv_init_uniform_shaped(b200conv_t* h, size_t block, const float* const* raw, size_t n, const b200conv_ir_shape_params* sp) {
  REQUIRE_CUDA(h);
  const size_t off = 0;
  return init_shaped(h, 1, &block, &off, raw, n, sp);
}

int b200conv_init_twostage_shaped(b200conv_t* h, size_t head_block, size_t tail_block, const float* const* raw, size_t n,
                                  const b200conv_ir_shape_params* sp) {
  REQUIRE_CUDA(h);
  if (head_block == 0 || tail_block == 0) return fail(h, B200CONV_EINVAL, "block size 0");
  if (head_block > tail_block) std::swap(head_block, tail_block);
  const size_t hb = next_pow2(head_block), tb = next_pow2(tail_block);
  const size_t blocks[2] = {hb, tb};
  const size_t offsets[2] = {0, 2 * tb};
  return init_shaped(h, 2, blocks, offsets, raw, n, sp);
}

int b200conv_process_device(b200conv_t* h, const float* in_dev, size_t in_stride,
                            float* out_dev, size_t out_stride, size_t len, int sync) {
  REQUIRE_CUDA(h);
  if (int rc = set_device(h)) return rc;
  if (h->timing) h->ev_used = 0;
  if (h->stages.empty()) {      // no IR: zeros (FFTConvolver.cpp:157-161)
    if (len) CU_CHECK(h, cudaMemset2DAsync(out_dev, out_stride * sizeof(float), 0, len * sizeof(float),
                                           h->route_on ? h->n_out : h->C, h->s_main));
  } else {
    const size_t B0 = h->stages[0].B;
    const size_t chunk = h->Lmax - B0;     // keeps fill + n <= Lmax for every stage (inbuf holds B + Lmax samples)
    const bool overlap = len > chunk || h->cfg.shard_count > 1;    // (slot-exchange groups always use s_post)
    size_t done = 0;
    if (const int nc = rt_cluster_ctas(h, len)) {       // a call inside the open block: one cluster kernel
      if (int rc = rt_call(h, nc, in_dev, in_stride, out_dev, out_stride, len, false)) return rc;
      done = len;
    }
    while (done < len) {
      size_t n = std::min(len - done, chunk);
      if (int rc = run_group(h, in_dev + done, in_stride, out_dev + done, out_stride, n, overlap)) return rc;
      done += n;
    }
    if (overlap) { if (int rc = join_post(h)) return rc; }
  }
  if (sync || h->timing) {
    CU_CHECK(h, cudaStreamSynchronize(h->s_main));
    if (h->timing) timing_collect(h);
    if (int rc = p2p_check(h)) return rc;
  }
  return B200CONV_OK;
}

// Host -> device staging of one launch group (n samples per channel from in[c] + off into din[b], channel pitch
// `pitch`) on stream st.  With the slot exchange's input broadcast only shard 0 touches PCIe: it uploads the
// group, stores it into every peer's din[b] over NVLink and an "input landed" flag barrier releases the peers.
// Launch-group sizes of a pipelined host-pointer call: the H2D copy of the FIRST group and the D2H copy of the LAST one
// cannot overlap with compute, so the sequence ramps up from one sweep wave (w, 2w, 4w, ...), runs steady groups of
// `grp` samples and ramps down again; every group but the last is a whole number of waves / 64-block tiles, the last
// one carries whatever is left (incl. a ragged tail).
static std::vector<size_t> ramped_groups(size_t len, size_t wave, size_t tile, size_t grp, size_t cap) {
  std::vector<size_t> g, up;
  size_t tot = 0;
  for (size_t r = wave; r * 2 <= grp && 2 * (tot + r) + 2 * grp <= len; r *= 2) { up.push_back(r); tot += r; }
  size_t remaining = len;
  for (size_t r : up) { g.push_back(r); remaining -= r; }
  while (remaining > tot + grp) { g.push_back(grp); remaining -= grp; }
  if (!up.empty()) {
    const size_t mid = (remaining - tot) / tile * tile;
    if (mid) { g.push_back(mid); remaining -= mid; }
    for (size_t i = up.size(); i-- > 1;) { g.push_back(up[i]); remaining -= up[i]; }
  }
  if (remaining) g.push_back(remaining);
  std::vector<size_t> out;                      // no group above the staging capacity
  for (size_t v : g) { while (v > cap) { out.push_back(cap); v -= cap; } if (v) out.push_back(v); }
  return out;
}

static int stage_input(b200conv_t* h, int b, const float* const* in, size_t off, size_t n, size_t pitch, int Cin,
                       const float* packed_src, cudaStream_t st) {
  const bool bc = h->p2p_on && h->bcast_in;
  if (!bc || h->cfg.shard_rank == 0) {
    if (packed_src) {
      CU_CHECK(h, cudaMemcpyAsync(h->din[b], packed_src, (size_t)Cin * n * sizeof(float), cudaMemcpyHostToDevice, st));
    } else {
      for (int c = 0; c < Cin; ++c)
        CU_CHECK(h, cudaMemcpyAsync(h->din[b] + (size_t)c * pitch, in[c] + off, n * sizeof(float), cudaMemcpyHostToDevice, st));
    }
  }
  if (bc) {
    if (h->cfg.shard_rank == 0) {
      // the peers read din[b] in the forward FFT of the group two exchange groups ago: its first barrier has passed
      CU_CHECK(h, cudaStreamWaitEvent(st, h->ev_b1[h->xgrp & 1], 0));
      for (int r = 1; r < h->cfg.shard_count; ++r)
        if (int rc = copy_rows_kernel(h, h->peer_din[r][b], pitch, h->din[b], pitch, n, Cin, st)) return rc;
    }
    if (int rc = p2p_barrier(h, st, 1)) return rc;
  }
  return 0;
}

static int process_impl(b200conv_t* h, const float* const* in, float* const* out_user, size_t len) {
  REQUIRE_CUDA(h);
  if (len == 0) return B200CONV_OK;
  if (!in) return fail(h, B200CONV_EINVAL, "null buffer");
  // only shard 0 of a sharded handle produces audio; the other shards leave `out` untouched (no D2H, and
  // no host memset either: that would cost more than the whole step on the throughput path)
  float* const* out = (out_user && h->cfg.shard_rank != 0) ? nullptr : out_user;
  if (int rc = set_device(h)) return rc;
  if (h->timing) h->ev_used = 0;
  const int C = h->C;
  const int Cin = h->route_on ? h->n_in : C, Cout = h->route_on ? h->n_out : C;
  if (h->stages.empty()) {
    if (out) for (int c = 0; c < Cout; ++c) std::memset(out[c], 0, len * sizeof(float));
    return B200CONV_OK;
  }
  const size_t B0 = h->stages[0].B;
  const size_t chunk = h->Lmax - B0;
  if (len <= chunk && len <= std::max((size_t)64 * B0, (size_t)16384)) {
    if (const int nc = (len <= h->hpin_cap && h->hpin_in_dev && h->hpin_out_dev) ? rt_cluster_ctas(h, len) : 0) {
      // real-time path: the cluster kernel reads the samples straight from the pinned staging buffer and writes the
      // result into it (zero-copy over PCIe): one launch + one synchronise per call
      for (int c = 0; c < Cin; ++c) std::memcpy(h->hpin_in + (size_t)c * len, in[c], len * sizeof(float));
      if (int rc = rt_call(h, nc, h->hpin_in_dev, len, h->hpin_out_dev, len, len, true)) return rc;
      // wait for the kernel's completion word (set after all output stores) instead of the driver's stream
      // synchronise; if it does not show up within 20 ms, fall back to the synchronise (and its error report)
      bool done = false;
      if (h->hflag_dev) {
        volatile unsigned int* f = h->hflag;
        const unsigned int want = h->flag_epoch;
        const auto t0 = std::chrono::steady_clock::now();
        for (unsigned spins = 0; !(done = (*f == want)); ++spins)
          if ((spins & 0x3ff) == 0x3ff &&
              std::chrono::steady_clock::now() - t0 > std::chrono::milliseconds(20)) break;
      }
      if (!done) CU_CHECK(h, cudaStreamSynchronize(h->s_main));
      if (out)
        for (int c = 0; c < Cout; ++c) std::memcpy(out[c], h->hpin_out + (size_t)c * len, len * sizeof(float));
      return B200CONV_OK;
    }
    // latency path: one stream, one group; all channels travel in ONE pinned H2D and ONE D2H copy
    // (channel pitch = len), which matters for the 2-4 channel handles of a StereoConvolver
    const bool packed = len <= h->hpin_cap;
    const size_t pitch = packed ? len : h->Lmax;
    const bool uploads = !(h->p2p_on && h->bcast_in) || h->cfg.shard_rank == 0;
    if (packed && uploads)
      for (int c = 0; c < Cin; ++c) std::memcpy(h->hpin_in + (size_t)c * len, in[c], len * sizeof(float));
    if (int rc = stage_input(h, 0, in, 0, len, pitch, Cin, packed ? h->hpin_in : nullptr, h->s_main)) return rc;
    const bool ov = h->cfg.shard_count > 1;
    if (int rc = run_group(h, h->din[0], pitch, h->dout[0], pitch, len, ov)) return rc;
    if (ov) { if (int rc = join_post(h)) return rc; }
    if (out) {
      if (packed) {
        CU_CHECK(h, cudaMemcpyAsync(h->hpin_out, h->dout[0], (size_t)Cout * len * sizeof(float), cudaMemcpyDeviceToHost, h->s_main));
      } else {
        for (int c = 0; c < Cout; ++c)
          CU_CHECK(h, cudaMemcpyAsync(out[c], h->dout[0] + (size_t)c * h->Lmax, len * sizeof(float), cudaMemcpyDeviceToHost, h->s_main));
      }
    }
    CU_CHECK(h, cudaStreamSynchronize(h->s_main));
    if (out && packed)
      for (int c = 0; c < Cout; ++c) std::memcpy(out[c], h->hpin_out + (size_t)c * len, len * sizeof(float));
    return p2p_check(h);
  }
  // throughput path: H2D / compute / D2H of successive groups overlap on three streams
  size_t done = 0;
  int i = 0;
  // Split long calls into groups so that the PCIe copies overlap with compute: only the first group's H2D
  // and the last group's D2H are exposed, so aim for ~8 groups — but keep every group a whole number of
  // sweep WAVES (n_sm x 3 CTAs x 64 blocks per CTA over ceil(B/32) x C tile columns), otherwise a
  // partially filled last wave costs more than the overlap gains.
  const size_t tile = (size_t)B0 * 64;
  const size_t cols = (size_t)((B0 + 31) / 32) * (size_t)h->C;
  size_t wave = ((size_t)h->n_sm * 3 * 64 + cols - 1) / cols * (size_t)B0;       // samples per full wave
  wave = std::max(tile, wave / tile * tile);
  size_t grp = std::max(wave, (len / 8) / wave * wave);
  grp = std::min(grp, chunk >= tile ? chunk / tile * tile : chunk);
  const std::vector<size_t> groups = ramped_groups(len, wave, tile, grp, chunk);
  for (size_t gi = 0; gi < groups.size() && done < len; ++gi, ++i) {
    const int b = i & 1;
    const size_t n = std::min(len - done, groups[gi]);
    if (i >= 2) CU_CHECK(h, cudaStreamWaitEvent(h->s_in, h->ev_din[b], 0));     // din[b] free again
    if (int rc = stage_input(h, b, in, done, n, h->Lmax, Cin, nullptr, h->s_in)) return rc;
    CU_CHECK(h, cudaEventRecord(h->ev_h2d[b], h->s_in));
    CU_CHECK(h, cudaStreamWaitEvent(h->s_main, h->ev_h2d[b], 0));
    if (i >= 2) CU_CHECK(h, cudaStreamWaitEvent(h->s_post, h->ev_d2h[b], 0));    // dout[b] drained
    if (int rc = run_group(h, h->din[b], h->Lmax, h->dout[b], h->Lmax, n, true)) return rc;
    CU_CHECK(h, cudaEventRecord(h->ev_din[b], h->s_main));    // every read of din[b] is queued on s_main
    CU_CHECK(h, cudaEventRecord(h->ev_comp[b], h->s_post));    // dout[b] complete
    CU_CHECK(h, cudaStreamWaitEvent(h->s_out, h->ev_comp[b], 0));
    if (out)
      for (int c = 0; c < Cout; ++c)
        CU_CHECK(h, cudaMemcpyAsync(out[c] + done, h->dout[b] + (size_t)c * h->Lmax, n * sizeof(float), cudaMemcpyDeviceToHost, h->s_out));
    CU_CHECK(h, cudaEventRecord(h->ev_d2h[b], h->s_out));
    done += n;
  }
  CU_CHECK(h, cudaStreamSynchronize(h->s_out));
  if (int rc = join_post(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  return p2p_check(h);
}

int b200conv_process(b200conv_t* h, const float* const* in, float* const* out, size_t len) {
  if (h && len && !out) return fail(h, B200CONV_EINVAL, "null buffer");
  return process_impl(h, in, out, len);
}

int b200conv_prime(b200conv_t* h, const float* const* in, size_t len) { return process_impl(h, in, nullptr, len); }

int b200conv_process_device_sliced(b200conv_t* h, const float* in_dev, size_t in_stride, float* out_dev, size_t out_stride,
                                   size_t len, int slice_rank, int slice_count, int sync) {
  REQUIRE_CUDA(h);
  if (int rc = set_device(h)) return rc;
  if (h->timing) h->ev_used = 0;
  if (h->stages.empty()) {
    if (len) CU_CHECK(h, cudaMemset2DAsync(out_dev, out_stride * sizeof(float), 0, len * sizeof(float), h->C, h->s_main));
  } else {
    SlicePlan sp;
    if (int rc = plan_slice(h, len, slice_rank, slice_count, &sp)) return rc;
    Stage& s = h->stages[0];
    const size_t B = (size_t)s.B;
    const long long done0 = s.blocks_done, pos0 = h->abs_pos;
    if (int rc = advance_fft_only(h, in_dev + (size_t)sp.lo * B, in_stride, sp.a - sp.lo)) return rc;
    const size_t chunk = (h->Lmax - B) / B * B;
    const size_t n_slice = (size_t)(sp.b - sp.a) * B;
    const bool overlap = n_slice > chunk;
    for (size_t done = 0; done < n_slice;) {
      const size_t n = std::min(n_slice - done, chunk);
      const size_t off = (size_t)sp.a * B + done;
      if (int rc = run_group(h, in_dev + off, in_stride, out_dev + off, out_stride, n, overlap)) return rc;
      done += n;
    }
    if (overlap) { if (int rc = join_post(h)) return rc; }
    if (int rc = advance_fft_only(h, in_dev + (size_t)sp.tail_lo * B, in_stride, sp.T - sp.tail_lo)) return rc;
    s.blocks_done = done0 + sp.T;               // the state is that of the whole call
    h->abs_pos = pos0 + (long long)len;
  }
  if (sync || h->timing) {
    CU_CHECK(h, cudaStreamSynchronize(h->s_main));
    if (h->timing) timing_collect(h);
  }
  return B200CONV_OK;
}

int b200conv_process_sliced(b200conv_t* h, const float* const* in, float* const* out, size_t len, int slice_rank, int slice_count) {
  REQUIRE_CUDA(h);
  if (len == 0) return B200CONV_OK;
  if (!in || !out) return fail(h, B200CONV_EINVAL, "null buffer");
  if (int rc = set_device(h)) return rc;
  if (h->timing) h->ev_used = 0;
  const int C = h->C;
  if (h->stages.empty()) {                      // no IR: zeros (FFTConvolver.cpp:157-161); every GPU writes the same value
    for (int c = 0; c < C; ++c) std::memset(out[c], 0, len * sizeof(float));
    return B200CONV_OK;
  }
  SlicePlan sp;
  if (int rc = plan_slice(h, len, slice_rank, slice_count, &sp)) return rc;
  Stage& s = h->stages[0];
  const size_t B = (size_t)s.B;
  const long long done0 = s.blocks_done, pos0 = h->abs_pos;
  // pieces of at most `grp` samples, each one H2D -> (forward FFTs | full group) -> D2H, pipelined over the three
  // streams like b200conv_process: [lo, a) and [tail_lo, T) are transformed only, [a, b) is convolved
  const size_t chunk = (h->Lmax - B) / B * B;
  const size_t tile = B * 64;
  const size_t cols = (size_t)((B + 31) / 32) * (size_t)C;
  size_t wave = ((size_t)h->n_sm * 3 * 64 + cols - 1) / cols * B;
  wave = std::max(tile, wave / tile * tile);
  const size_t n_slice = (size_t)(sp.b - sp.a) * B;
  size_t grp = std::max(wave, (n_slice / 4) / wave * wave);
  grp = std::min(grp, chunk >= tile ? chunk / tile * tile : chunk);
  struct Piece { size_t off, n; bool conv; };
  std::vector<Piece> pieces;
  auto add = [&](long long b0, long long b1, bool conv) {
    for (size_t o = (size_t)b0 * B, e = (size_t)b1 * B; o < e; o += grp) pieces.push_back({o, std::min(grp, e - o), conv});
  };
  add(sp.lo, sp.a, false);
  {   // the slice itself: ramped groups (short first H2D, short last D2H)
    size_t o = (size_t)sp.a * B;
    for (size_t gsz : ramped_groups(n_slice, wave, tile, grp, chunk)) { pieces.push_back({o, gsz, true}); o += gsz; }
  }
  add(sp.tail_lo, sp.T, false);
  int i = 0;
  bool used_out[2] = {false, false};
  for (const Piece& pc_ : pieces) {
    const int b = i & 1;
    if (i >= 2) CU_CHECK(h, cudaStreamWaitEvent(h->s_in, h->ev_din[b], 0));
    for (int c = 0; c < C; ++c)
      CU_CHECK(h, cudaMemcpyAsync(h->din[b] + (size_t)c * h->Lmax, in[c] + pc_.off, pc_.n * sizeof(float), cudaMemcpyHostToDevice, h->s_in));
    CU_CHECK(h, cudaEventRecord(h->ev_h2d[b], h->s_in));
    CU_CHECK(h, cudaStreamWaitEvent(h->s_main, h->ev_h2d[b], 0));
    if (!pc_.conv) {
      if (int rc = advance_fft_only(h, h->din[b], h->Lmax, (long long)(pc_.n / B))) return rc;
      CU_CHECK(h, cudaEventRecord(h->ev_din[b], h->s_main));
    } else {
      if (used_out[b]) CU_CHECK(h, cudaStreamWaitEvent(h->s_post, h->ev_d2h[b], 0));
      if (int rc = run_group(h, h->din[b], h->Lmax, h->dout[b], h->Lmax, pc_.n, true)) return rc;
      CU_CHECK(h, cudaEventRecord(h->ev_din[b], h->s_main));
      CU_CHECK(h, cudaEventRecord(h->ev_comp[b], h->s_post));
      CU_CHECK(h, cudaStreamWaitEvent(h->s_out, h->ev_comp[b], 0));
      for (int c = 0; c < C; ++c)
        CU_CHECK(h, cudaMemcpyAsync(out[c] + pc_.off, h->dout[b] + (size_t)c * h->Lmax, pc_.n * sizeof(float), cudaMemcpyDeviceToHost, h->s_out));
      CU_CHECK(h, cudaEventRecord(h->ev_d2h[b], h->s_out));
      used_out[b] = true;
    }
    ++i;
  }
  CU_CHECK(h, cudaStreamSynchronize(h->s_out));
  if (int rc = join_post(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  s.blocks_done = done0 + sp.T;
  h->abs_pos = pos0 + (long long)len;
  return B200CONV_OK;
}

int b200conv_register_host(void* p, size_t bytes) {
#if defined(PC_EMULATE)
  (void)p; (void)bytes;
  return B200CONV_OK;
#else
  if (cudaHostRegister(p, bytes, cudaHostRegisterPortable) != cudaSuccess) { cudaGetLastError(); return B200CONV_ECUDA; }
  return B200CONV_OK;
#endif
}

int b200conv_unregister_host(void* p) {
#if defined(PC_EMULATE)
  (void)p;
  return B200CONV_OK;
#else
  if (cudaHostUnregister(p) != cudaSuccess) { cudaGetLastError(); return B200CONV_ECUDA; }
  return B200CONV_OK;
#endif
}

int b200conv_process_xfade(b200conv_t* ho, b200conv_t* hn, const float* const* in, float* const* out,
                           size_t len, float alpha0, float alpha_step) {
  REQUIRE_CUDA(ho);
  REQUIRE_CUDA(hn);
  if (len == 0) return B200CONV_OK;
  if (!in || !out) return fail(hn, B200CONV_EINVAL, "null buffer");
  if (ho == hn || ho->cfg.device != hn->cfg.device || ho->C != hn->C || ho->route_on != hn->route_on ||
      (ho->route_on && (ho->n_in != hn->n_in || ho->n_out != hn->n_out)) ||
      ho->cfg.shard_count > 1 || hn->cfg.shard_count > 1)
    return fail(hn, B200CONV_EINVAL, "crossfade needs two different unsharded handles with the same device, channels and routing");
  if (int rc = set_device(hn)) return rc;
  const int C = hn->C;
  const int Cin = hn->route_on ? hn->n_in : C, Cout = hn->route_on ? hn->n_out : C;
  if (ho->stages.empty() || hn->stages.empty()) {   // one side has no IR: its output is silence
    b200conv_t* live = ho->stages.empty() ? hn : ho;
    if (int rc = process_impl(live, in, out, len)) return rc;
    for (int c = 0; c < Cout; ++c)
      for (size_t i = 0; i < len; ++i) {
        const float al = std::fmin(1.0f, std::fmax(0.0f, alpha0 + alpha_step * (float)i));
        out[c][i] *= (live == hn) ? al : (1.0f - al);
      }
    return B200CONV_OK;
  }
#if !defined(PC_EMULATE)
  if (ho->Lmax != hn->Lmax) return fail(hn, B200CONV_EINVAL, "crossfade needs equal staging sizes (same head block and batch size)");
#endif
  if (ho->timing) ho->ev_used = 0;
  if (hn->timing) hn->ev_used = 0;
  const size_t chunk = std::min(ho->Lmax - ho->stages[0].B, hn->Lmax - hn->stages[0].B);
  for (size_t done = 0; done < len;) {
    const size_t n = std::min(len - done, chunk);
    // input once (old handle's staging), both convolvers read it
    for (int c = 0; c < Cin; ++c)
      CU_CHECK(ho, cudaMemcpyAsync(ho->din[0] + (size_t)c * ho->Lmax, in[c] + done, n * sizeof(float), cudaMemcpyHostToDevice, ho->s_main));
    CU_CHECK(ho, cudaEventRecord(ho->ev_h2d[0], ho->s_main));
    if (int rc = run_group(ho, ho->din[0], ho->Lmax, ho->dout[0], ho->Lmax, n, false)) return rc;
    CU_CHECK(ho, cudaEventRecord(ho->ev_comp[0], ho->s_main));
    CU_CHECK(hn, cudaStreamWaitEvent(hn->s_main, ho->ev_h2d[0], 0));
    if (int rc = run_group(hn, ho->din[0], ho->Lmax, hn->dout[0], hn->Lmax, n, false)) return rc;
    CU_CHECK(hn, cudaStreamWaitEvent(hn->s_main, ho->ev_comp[0], 0));
    const float a0 = alpha0 + alpha_step * (float)done;
#if defined(PC_EMULATE)
    for (int c = 0; c < Cout; ++c)
      for (size_t i = 0; i < n; ++i) {
        const float al = std::fmin(1.0f, std::fmax(0.0f, a0 + alpha_step * (float)i));
        float* d = hn->dout[0] + (size_t)c * hn->Lmax + i;
        *d = (1.0f - al) * ho->dout[0][(size_t)c * ho->Lmax + i] + al * *d;
      }
#else
    dim3 grid((unsigned)((n + 255) / 256), Cout, 1);
    pc::k_xfade<<<grid, 256, 0, hn->s_main>>>(hn->dout[0], ho->dout[0], hn->dout[0], (long long)hn->Lmax, (long long)n, a0, alpha_step);
    hn->launches++;
    CU_CHECK(hn, cudaGetLastError());
#endif
    for (int c = 0; c < Cout; ++c)
      CU_CHECK(hn, cudaMemcpyAsync(out[c] + done, hn->dout[0] + (size_t)c * hn->Lmax, n * sizeof(float), cudaMemcpyDeviceToHost, hn->s_main));
    CU_CHECK(hn, cudaStreamSynchronize(hn->s_main));
    done += n;
  }
  return B200CONV_OK;
}

// ---- send / wet chain (SURVEY 8f-4 + the rest of 8f-1) ------------------------------------------------------------
namespace {
// Filter::getCoeff (src/dsp/Filter.h:40-44): tan() through the reference's 2048-point lookup table with its cubic
// interpolation (src/dsp/Filter.h:28-36, src/dsp/Utils.h:50-112) — the coefficient has to be the reference's, bit for bit
float chain_coeff(float freq, float srate) {
  static float lut[2048];
  static std::once_flag once;
  std::call_once(once, [] {
    const float pi = 3.14159265358979323846f;
    for (int i = 0; i < 2048; ++i) {
      const float x = (float)i / 2047.0f;
      float mapped = 0.0f + x * (0.5f - 0.0f);
      mapped = std::min(std::max(mapped, 0.0f), 0.5f);
      const float max_rads = 0.499f * pi, scaled = mapped * pi;
      lut[i] = std::tan(std::min(max_rads, scaled));
    }
  });
  freq = std::min(std::max(freq, 20.0f), srate * 0.48f);
  float ratio = std::min(std::max(freq / srate, 0.0f), 0.5f);
  const float scaler = 2047.0f / 0.5f;
  const float index = ratio * scaler + 0.0f;
  const int i = (int)index;
  const float t = index - (float)i;
  const int i0 = std::max(0, i - 1), i1 = i, i2 = std::min(2047, i + 1), i3 = std::min(2047, i + 2);
  const float y0 = lut[i0], y1 = lut[i1], y2 = lut[i2], y3 = lut[i3];
  const float a0 = y3 - y2 - y0 + y1, a1 = y0 - y1 - a0, a2 = y2 - y0, a3 = y1;
  return (a0 * t * t * t) + (a1 * t * t) + (a2 * t) + a3;
}

// Filter::init (src/dsp/Filter.cpp:3-21) with the q the processor passes (src/PluginProcessor.cpp:845-848)
pc::ChainFilter chain_filter(bool on, int slope, int mode, float srate, float freq) {
  pc::ChainFilter f{};
  f.on = on ? 1 : 0; f.slope = slope; f.mode = mode;
  const float q = slope == 2 ? 0.0765f : 0.2929f, q2 = 0.6173f;
  f.g = chain_coeff(freq, srate);
  f.k = 2 - 2 * q;
  f.k2 = 2 - 2 * q2;
  if (slope == 0) {
    f.g = f.g / (1.0f + f.g);
  } else {
    f.a1 = 1.0f / (1.0f + f.g * (f.g + f.k));
    f.a2 = f.g * f.a1;
    f.a3 = f.g * f.a2;
    f.a12 = 1.0f / (1.0f + f.g * (f.g + f.k2));
    f.a22 = f.g * f.a12;
    f.a32 = f.g * f.a22;
  }
  return f;
}
}  // namespace

int b200conv_chain_configure(b200conv_t* h, const b200conv_chain_config* cfg) {
  REQUIRE_CUDA(h);
  if (!cfg) { h->chain_on = false; h->route_in_only = false; return B200CONV_OK; }
  if (h->C != 2 && h->C != 4) return fail(h, B200CONV_ESTATE, "the send / wet chain needs a stereo (C = 2) or quad (C = 4) handle");
  if (h->route_on) return fail(h, B200CONV_ESTATE, "the send / wet chain cannot be combined with b200conv_set_routing");
  if (h->cfg.shard_count != 1) return fail(h, B200CONV_ESTATE, "the send / wet chain needs an unsharded handle");
  if (h->stages.empty()) return fail(h, B200CONV_ESTATE, "load an impulse response first");
  if (cfg->srate <= 0 || cfg->predelay < 0 || cfg->lowcut_slope < 0 || cfg->lowcut_slope > 2 || cfg->highcut_slope < 0 || cfg->highcut_slope > 2)
    return fail(h, B200CONV_EINVAL, "bad chain configuration");
  if (int rc = set_device(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  h->chain_cfg = *cfg;
  const float sr = (float)cfg->srate;
  h->chain_lc = chain_filter(cfg->lowcut_hz > 20.0f, cfg->lowcut_slope, 2, sr, cfg->lowcut_hz);          // HP, PluginProcessor.cpp:1643
  h->chain_hc = chain_filter(cfg->highcut_hz < 20000.0f, cfg->highcut_slope, 0, sr, cfg->highcut_hz);   // LP, :1647
  const size_t L = h->Lmax;
  const size_t ring = next_pow2((size_t)cfg->predelay + L + 1);
  if (!h->c_io) {
    CU_CHECK(h, cudaMalloc(&h->c_io, 6 * L * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&h->c_conv_in, 2 * L * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&h->c_filt, 2 * L * sizeof(float)));
    CU_CHECK(h, cudaMalloc(&h->c_state, 2 * pc::kChainStates * sizeof(float)));
    CU_CHECK(h, cudaMallocHost((void**)&h->c_hpin, 6 * h->hpin_cap * sizeof(float)));
#if defined(PC_EMULATE)
    h->c_hpin_dev = h->c_hpin;
#else
    if (cudaHostGetDevicePointer((void**)&h->c_hpin_dev, h->c_hpin, 0) != cudaSuccess) { cudaGetLastError(); h->c_hpin_dev = nullptr; }
#endif
  }
  if (ring != h->c_ring_size) {
    cudaFree(h->c_ring); h->c_ring = nullptr;
    CU_CHECK(h, cudaMalloc(&h->c_ring, 2 * ring * sizeof(float)));
    h->c_ring_size = ring;
  }
  // Filter::reset(0) + cleared delay line (src/PluginProcessor.cpp:654-657)
  CU_CHECK(h, cudaMemsetAsync(h->c_state, 0, 2 * pc::kChainStates * sizeof(float), h->s_main));
  CU_CHECK(h, cudaMemsetAsync(h->c_ring, 0, 2 * ring * sizeof(float), h->s_main));
  h->c_ring_pos = 0;
  for (int c = 0; c < 8; ++c) h->in_map[c] = c & 1;        // LL, RR, LR, RL <- L, R, L, R (StereoConvolver.cpp:35-40)
  h->chain_on = true;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  return B200CONV_OK;
}

int b200conv_chain_process(b200conv_t* h, const float* const* dry, const float* ysend, const float* yrev, float* const* out, size_t len) {
  REQUIRE_CUDA(h);
  if (len == 0) return B200CONV_OK;
  if (!h->chain_on) return fail(h, B200CONV_ESTATE, "b200conv_chain_configure first");
  if (!dry || !out || !dry[0] || !dry[1] || !out[0] || !out[1]) return fail(h, B200CONV_EINVAL, "null buffer");
  if (h->stages.empty()) return fail(h, B200CONV_ESTATE, "no impulse response loaded");
  if (int rc = set_device(h)) return rc;
  const int C = h->C;
  const size_t L = h->Lmax, B0 = h->stages[0].B;
  const size_t chunk = L - B0;
  float* d_dry = h->c_io; float* d_send = h->c_io + 2 * L; float* d_rev = h->c_io + 3 * L; float* d_out = h->c_io + 4 * L;
  // real-time calls: the kernels read the dry block + envelopes straight from pinned host memory and write the mix
  // back into it (zero-copy), so a callback is three launches and one synchronise instead of six copies more
  const bool zc = len <= h->hpin_cap && len <= chunk && h->c_hpin_dev != nullptr && h->opt_rt;
  size_t dstride = L;
  if (zc) {
    const size_t cap = h->hpin_cap;
    std::memcpy(h->c_hpin, dry[0], len * sizeof(float));
    std::memcpy(h->c_hpin + cap, dry[1], len * sizeof(float));
    if (ysend) std::memcpy(h->c_hpin + 2 * cap, ysend, len * sizeof(float));
    if (yrev) std::memcpy(h->c_hpin + 3 * cap, yrev, len * sizeof(float));
    d_dry = h->c_hpin_dev; d_send = h->c_hpin_dev + 2 * cap; d_rev = h->c_hpin_dev + 3 * cap; d_out = h->c_hpin_dev + 4 * cap;
    dstride = cap;
  }
  for (size_t done = 0; done < len;) {
    const size_t n = std::min(len - done, chunk);
    if (!zc) {
      for (int ch = 0; ch < 2; ++ch)
        CU_CHECK(h, cudaMemcpyAsync(d_dry + ch * L, dry[ch] + done, n * sizeof(float), cudaMemcpyHostToDevice, h->s_main));
      if (ysend) CU_CHECK(h, cudaMemcpyAsync(d_send, ysend + done, n * sizeof(float), cudaMemcpyHostToDevice, h->s_main));
      if (yrev) CU_CHECK(h, cudaMemcpyAsync(d_rev, yrev + done, n * sizeof(float), cudaMemcpyHostToDevice, h->s_main));
    }
    pc::ChainSendParams sp{};
    sp.dry = d_dry; sp.dry_stride = (long long)dstride; sp.ysend = ysend ? d_send : nullptr;
    sp.conv_in = h->c_conv_in; sp.conv_stride = (long long)L;
    sp.filt = h->c_filt; sp.filt_stride = (long long)L;
    sp.state = h->c_state;
    sp.ring = h->c_ring; sp.ring_stride = (long long)h->c_ring_size; sp.ring_mask = (long long)h->c_ring_size - 1;
    sp.ring_pos = h->c_ring_pos; sp.predelay = h->chain_cfg.predelay; sp.n = (long long)n;
    sp.lc = h->chain_lc; sp.hc = h->chain_hc;
    // chunks: two passes of n/T sequential samples (~200 cycles each) + a serial scan of T 8x8 matrix-vector steps
    // (~256 cycles each): T ~ sqrt(1.5 n), a power of two in [8, 1024]
    int T = 8;
    while (T < 1024 && (size_t)T * T < n + n / 2) T *= 2;
#if defined(PC_EMULATE)
    pc::emu_chain_send(sp, T);
#else
    pc::k_chain_send<<<2, T, 0, h->s_main>>>(sp);
    CU_CHECK(h, cudaGetLastError());
#endif
    h->launches++;
    h->c_ring_pos = (h->c_ring_pos + (long long)n) & ((long long)h->c_ring_size - 1);
    // the convolvers: LL, RR[, LR, RL] read the chain's L / R, per-convolver outputs stay on the device
    h->route_in_only = true;
    int rc = 0;
    if (const int nc = rt_cluster_ctas(h, n)) rc = rt_call(h, nc, h->c_conv_in, L, h->dch[0], L, n, false);
    else rc = run_group(h, h->c_conv_in, L, h->dch[0], L, n, false);
    h->route_in_only = false;
    if (rc) return rc;
    pc::ChainWetParams wp{};
    wp.dry = d_dry; wp.dry_stride = (long long)dstride;
    wp.conv = h->dch[0]; wp.conv_stride = (long long)L;
    wp.yrev = yrev ? d_rev : nullptr;
    wp.out = d_out; wp.out_stride = (long long)dstride; wp.n = (long long)n;
    wp.quad_ts = (C == 4 && h->chain_cfg.true_stereo) ? 1 : 0;
    wp.width = h->chain_cfg.width; wp.drygain = h->chain_cfg.drygain; wp.wetgain = h->chain_cfg.wetgain;
#if defined(PC_EMULATE)
    pc::emu_chain_wet(wp);
#else
    pc::k_chain_wet<<<(unsigned)((n + 255) / 256), 256, 0, h->s_main>>>(wp);
    CU_CHECK(h, cudaGetLastError());
#endif
    h->launches++;
    if (!zc)
      for (int ch = 0; ch < 2; ++ch)
        CU_CHECK(h, cudaMemcpyAsync(out[ch] + done, d_out + ch * L, n * sizeof(float), cudaMemcpyDeviceToHost, h->s_main));
    CU_CHECK(h, cudaStreamSynchronize(h->s_main));
    if (zc)
      for (int ch = 0; ch < 2; ++ch) std::memcpy(out[ch], h->c_hpin + (4 + ch) * h->hpin_cap, n * sizeof(float));
    done += n;
  }
  return B200CONV_OK;
}

int b200conv_clear(b200conv_t* h) {
  REQUIRE_CUDA(h);
  if (int rc = set_device(h)) return rc;
  if (int rc = clear_state(h)) return rc;
  if (h->chain_on) {            // the chain's own history goes with the convolver's
    CU_CHECK(h, cudaMemsetAsync(h->c_state, 0, 2 * pc::kChainStates * sizeof(float), h->s_main));
    CU_CHECK(h, cudaMemsetAsync(h->c_ring, 0, 2 * h->c_ring_size * sizeof(float), h->s_main));
    h->c_ring_pos = 0;
  }
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  return p2p_check(h);
}

int b200conv_reset(b200conv_t* h) {
  REQUIRE_CUDA(h);
  if (int rc = set_device(h)) return rc;
  CU_CHECK(h, cudaStreamSynchronize(h->s_main));
  CU_CHECK(h, cudaStreamSynchronize(h->s_post));
  if (h->s_tail) CU_CHECK(h, cudaStreamSynchronize(h->s_tail));
  free_all(h);
  return B200CONV_OK;
}

int b200conv_num_stages(const b200conv_t* h) { return h ? (int)h->stages.size() : 0; }

int b200conv_stage(const b200conv_t* h, int s, b200conv_stage_info* out) {
  if (!h || !out || s < 0 || s >= (int)h->stages.size()) return B200CONV_EINVAL;
  const Stage& st = h->stages[s];
  out->block = st.B; out->partitions = st.P_full; out->tap_offset = st.tap_off;
  out->p_begin = st.p_begin; out->p_end = st.p_end;
  return B200CONV_OK;
}

size_t b200conv_ir_len(const b200conv_t* h, int channel) {
  if (!h || channel < 0 || channel >= h->C) return 0;
  return h->ir_len[channel];
}

unsigned long long b200conv_launch_count(const b200conv_t* h) { return h ? h->launches : 0; }

int b200conv_last_sweep_variant(const b200conv_t* h) { return h ? h->last_variant : 0; }

int b200conv_set_option(b200conv_t* h, const char* name, int value) {
  if (!h || !name) return B200CONV_EINVAL;
  const std::string n(name);
  if (n == "rt") h->opt_rt = value != 0;
  else if (n == "fft512") h->opt_fft512 = value != 0;
  else if (n == "slice_keep_tail") h->opt_slice_tail = value != 0;
  else if (n == "stream_alternate") h->opt_stream_alt = value != 0;
  else if (n == "tc") h->opt_tc = value != 0;
  else if (n == "tfft") h->opt_tfft = value != 0;
  else return fail(h, B200CONV_EINVAL, "unknown option");
  return B200CONV_OK;
}

int b200conv_set_timing(b200conv_t* h, int enable) {
  if (!h) return B200CONV_EINVAL;
  h->timing = enable != 0;
  return B200CONV_OK;
}

int b200conv_last_timing(const b200conv_t* h, float* cmac_ms, float* fft_ms, float* ifft_ms, int* cmac_launches) {
  if (!h) return B200CONV_EINVAL;
  if (cmac_ms) *cmac_ms = h->t_cmac;
  if (fft_ms) *fft_ms = h->t_fft;
  if (ifft_ms) *ifft_ms = h->t_ifft;
  if (cmac_launches) *cmac_launches = h->n_cmac;
  return B200CONV_OK;
}

void* b200conv_stream(const b200conv_t* h) { return h ? (void*)h->s_main : nullptr; }

int b200conv_set_reduce(b200conv_t* h, b200conv_reduce_fn fn, void* user) {
  if (!h) return B200CONV_EINVAL;
  h->reduce = fn; h->reduce_user = user;
  return B200CONV_OK;
}

int b200conv_set_routing(b200conv_t* h, int n_in, const int* in_map, int n_out, const float* mix) {
  if (!h) return B200CONV_EINVAL;
  if (n_in == 0) { h->route_on = false; return B200CONV_OK; }
  if (h->chain_on) return fail(h, B200CONV_ESTATE, "routing cannot be combined with the send / wet chain");
  const int C = h->C;
  if (C > 8 || n_in < 1 || n_in > C || n_out < 1 || n_out > C || !in_map || !mix)
    return fail(h, B200CONV_EINVAL, "routing needs C <= 8, 1 <= n_in, n_out <= C, in_map[C] and mix[n_out*C]");
  for (int c = 0; c < C; ++c)
    if (in_map[c] < 0 || in_map[c] >= n_in) return fail(h, B200CONV_EINVAL, "in_map entry out of range");
  if (h->s_main) { cudaSetDevice(h->cfg.device); cudaStreamSynchronize(h->s_main); if (h->s_post) cudaStreamSynchronize(h->s_post); }
  h->n_in = n_in; h->n_out = n_out;
  for (int c = 0; c < 8; ++c) h->in_map[c] = c < C ? in_map[c] : 0;
  std::memset(h->mix, 0, sizeof(h->mix));
  for (int i = 0; i < n_out * C; ++i) h->mix[i] = mix[i];
  h->route_on = true;
  return B200CONV_OK;
}

size_t b200conv_p2p_blob_size(const b200conv_t* h) { (void)h; return sizeof(P2PRecord) * kP2PBuffers; }

static int p2p_export_impl(b200conv_t* h, void* blob, int mode);
static int p2p_import_impl(b200conv_t* h, const void* all_blobs);

// A failed export / import (CUDA IPC not permitted in this container, out of memory for the exchange
// buffers, ...) releases whatever was set up and leaves the handle usable on the reduce-hook path.
int b200conv_p2p_export(b200conv_t* h, void* blob, int mode) {
  REQUIRE_CUDA(h);
  const int rc = p2p_export_impl(h, blob, mode);
  if (rc != B200CONV_OK && rc != B200CONV_EINVAL && !h->sticky_cuda_error) { const std::string keep = h->err; p2p_release(h); h->err = keep; }
  return rc;
}

int b200conv_p2p_import(b200conv_t* h, const void* all_blobs) {
  REQUIRE_CUDA(h);
  const int rc = p2p_import_impl(h, all_blobs);
  if (rc != B200CONV_OK && !h->sticky_cuda_error) { const std::string keep = h->err; p2p_release(h); h->err = keep; }
  return rc;
}

static int p2p_export_impl(b200conv_t* h, void* blob, int mode) {
  if (!blob) return fail(h, B200CONV_EINVAL, "null blob");
  if (h->cfg.shard_count < 2 || h->cfg.shard_count > 8) return fail(h, B200CONV_ESTATE, "slot exchange needs 2..8 shards");
  if (h->stages.size() != 1) return fail(h, B200CONV_ESTATE, "slot exchange supports uniform (single-stage) handles");
  if (int rc = set_device(h)) return rc;
  if (int rc = p2p_alloc(h)) return rc;
  h->p2p_mode = mode;
  void* bufs[kP2PBuffers] = {h->Yx[0], h->Yx[1], h->Hh, h->xout[0], h->xout[1], h->xflags, h->din[0], h->din[1]};
  P2PRecord* rec = static_cast<P2PRecord*>(blob);
  for (int i = 0; i < kP2PBuffers; ++i) {
    std::memset(&rec[i], 0, sizeof(P2PRecord));
    rec[i].ptr = (unsigned long long)(uintptr_t)bufs[i];
#if defined(PC_EMULATE)
    rec[i].kind = 1;
#else
    if (mode == 1) {
      rec[i].kind = 1;
    } else {
      rec[i].kind = 2;
      cudaIpcMemHandle_t hd;
      CU_CHECK(h, cudaIpcGetMemHandle(&hd, bufs[i]));
      static_assert(sizeof(hd) == 64, "IPC handle size");
      std::memcpy(rec[i].ipc, &hd, 64);
    }
#endif
  }
  return B200CONV_OK;
}

static int p2p_import_impl(b200conv_t* h, const void* all_blobs) {
  if (!all_blobs || !h->Yx[0]) return fail(h, B200CONV_ESTATE, "export before import");
  if (int rc = set_device(h)) return rc;
  const int G = h->cfg.shard_count, me = h->cfg.shard_rank;
  const P2PRecord* rec = static_cast<const P2PRecord*>(all_blobs);
  for (int r = 0; r < G; ++r) {
    void* ptrs[kP2PBuffers];
    for (int i = 0; i < kP2PBuffers; ++i) {
      const P2PRecord& x = rec[r * kP2PBuffers + i];
      if (r == me || x.kind == 1) {
        ptrs[i] = (void*)(uintptr_t)x.ptr;
      } else {
#if defined(PC_EMULATE)
        return fail(h, B200CONV_EINVAL, "IPC records in the emulation build");
#else
        // only the buffers this shard touches are mapped: every peer's Yx + flags, shard 0's Hh + xout
        // (the din records, i >= 6, are only opened if the input broadcast gets enabled)
        const bool needed = (i <= 1) || (i == 5) || (r == 0 && i <= 4);
        ptrs[i] = nullptr;
        if (needed) {
          cudaIpcMemHandle_t hd;
          std::memcpy(&hd, x.ipc, 64);
          void* p = nullptr;
          CU_CHECK(h, cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
          h->ipc_opened.push_back(p);
          ptrs[i] = p;
        }
#endif
      }
    }
    h->peerYx[r][0] = static_cast<float2*>(ptrs[0]);
    h->peerYx[r][1] = static_cast<float2*>(ptrs[1]);
    h->peer_flags[r] = static_cast<unsigned int*>(ptrs[5]);
    h->peer_din[r][0] = (r == me || rec[r * kP2PBuffers + 6].kind == 1) ? static_cast<float*>(ptrs[6]) : nullptr;
    h->peer_din[r][1] = (r == me || rec[r * kP2PBuffers + 7].kind == 1) ? static_cast<float*>(ptrs[7]) : nullptr;
    if (r == 0) {
      h->peerHh0 = static_cast<float2*>(ptrs[2]);
      h->peer_xout0[0] = static_cast<float*>(ptrs[3]);
      h->peer_xout0[1] = static_cast<float*>(ptrs[4]);
    }
  }
  h->din_records.assign(reinterpret_cast<const unsigned char*>(all_blobs),
                        reinterpret_cast<const unsigned char*>(all_blobs) + (size_t)G * kP2PBuffers * sizeof(P2PRecord));
  h->p2p_on = true;
  return B200CONV_OK;
}

int b200conv_p2p_set_input_broadcast(b200conv_t* h, int enable) {
  if (!h) return B200CONV_EINVAL;
  if (enable && !h->p2p_on) return fail(h, B200CONV_ESTATE, "input broadcast needs an attached slot exchange");
#if !defined(PC_EMULATE)
  if (enable && h->cfg.shard_rank == 0) {      // map the peers' staging buffers now (cross-process: CUDA IPC)
    if (int rc = set_device(h)) return rc;
    const P2PRecord* rec = reinterpret_cast<const P2PRecord*>(h->din_records.data());
    for (int r = 1; r < h->cfg.shard_count; ++r)
      for (int i = 0; i < 2; ++i) {
        if (h->peer_din[r][i]) continue;
        const P2PRecord& x = rec[r * kP2PBuffers + 6 + i];
        cudaIpcMemHandle_t hd;
        std::memcpy(&hd, x.ipc, 64);
        void* p = nullptr;
        CU_CHECK(h, cudaIpcOpenMemHandle(&p, hd, cudaIpcMemLazyEnablePeerAccess));
        h->ipc_opened.push_back(p);
        h->peer_din[r][i] = static_cast<float*>(p);
      }
  }
#endif
  h->bcast_in = enable != 0;
  return B200CONV_OK;
}

int b200conv_p2p_detach(b200conv_t* h) {
  if (!h) return B200CONV_EINVAL;
  if (h->s_main) { cudaSetDevice(h->cfg.device); cudaStreamSynchronize(h->s_main); if (h->s_post) cudaStreamSynchronize(h->s_post); }
  const int rc = h->sticky_cuda_error ? B200CONV_OK : p2p_check(h);   // a barrier that gave up is reported here at the latest
  h->p2p_on = false;
  h->bcast_in = false;
  return rc;
}

int b200conv_p2p_set_host_barrier(b200conv_t* h, b200conv_barrier_fn fn, void* user) {
  if (!h) return B200CONV_EINVAL;
  h->host_barrier = fn; h->host_barrier_user = user;
  return B200CONV_OK;
}

#if defined(PC_EMULATE)
// tests/emu only: make the (n+1)-th device allocation from now fail once
void pc_emu_fail_malloc_after(int n) { g_emu_fail_malloc_in = n; }
#endif

void* b200conv_alloc_host(size_t bytes) {
  void* p = nullptr;
  if (cudaMallocHost(&p, bytes) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  return p;
}
void b200conv_free_host(void* p) { if (p) cudaFreeHost(p); }

}  // extern "C"
