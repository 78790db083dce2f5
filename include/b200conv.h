/*
 * b200conv.h — C ABI of the B200-native partitioned-convolution engine.
 *
 * Drop-in boundary for the hot path of tiagolr/reevr (REEV-R): everything behind
 *   fftconvolver::FFTConvolver::{init,process,clear,reset}          libs/FFTConvolver/FFTConvolver.h:62-80
 *   fftconvolver::TwoStageFFTConvolver::{init,process,reset,clear}  libs/FFTConvolver/TwoStageFFTConvolver.h:65-83
 *   StereoConvolver::{loadImpulse,process,reset,clear}              src/dsp/StereoConvolver.h:20-25
 * i.e. AudioFFT::fft/ifft (AudioFFT.h:135-158), ComplexMultiplyAccumulate / Sum (Utilities.h:319-344)
 * and the frequency-domain delay line they operate on.  Plain C: opaque handle, raw pointers
 * and sizes only, no C++/torch types, never throws.  One handle = C independent mono
 * convolvers ("channels", each with its own impulse response) that share the block schedule
 * and are processed by the same kernel launches (C = 1 reproduces one reference object;
 * C = 2 / 4 reproduces one StereoConvolver in stereo / quad mode).
 *
 * Status codes: 0 = ok, negative = error (message via b200conv_last_error).  There is NO CPU
 * fall-back: if CUDA is unavailable every call fails loudly with B200CONV_ECUDA.
 *
 * Threading contract = the reference's (FFTConvolver.h:44-47): one caller at a time per
 * handle; different handles are fully independent (own streams, own device arena).
 */
#ifndef B200CONV_H
#define B200CONV_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200CONV_OK        0
#define B200CONV_EINVAL   -1   /* bad argument (e.g. block size 0 — the reference's init()==false) */
#define B200CONV_ECUDA    -2   /* CUDA runtime error / no device */
#define B200CONV_ESTATE   -3   /* call not valid in this state */
#define B200CONV_ENOMEM   -4

typedef struct b200conv b200conv_t;

typedef struct b200conv_config {
  int n_channels;        /* C >= 1 mono convolvers in this handle                                  */
  int device;            /* CUDA device ordinal                                                     */
  int max_batch_blocks;  /* head-stage blocks processed per internal launch group (0 = default 4736) */
  int shard_rank;        /* partition-range shard owned by this handle (multi-GPU), 0 <= rank < n   */
  int shard_count;       /* number of shards (1 = unsharded)                                        */
  int cmac_variant;      /* 0 = auto; >0 selects a specific CMAC kernel variant (tuning/bench):     */
                         /* 22 packed-FMA batched, 40 tensor cores (tcgen05), 50..52 FFT along the */
                         /* block axis, 100..108 streaming                                         */
} b200conv_config;

/* Lifetime ------------------------------------------------------------------------------- */
b200conv_t* b200conv_create(const b200conv_config* cfg);     /* NULL only if cfg is invalid/OOM */
void        b200conv_destroy(b200conv_t* h);
const char* b200conv_last_error(const b200conv_t* h);         /* "" if none                      */

/* IR load (replaces FFTConvolver::init FFTConvolver.cpp:93-152 and
 * TwoStageFFTConvolver::init TwoStageFFTConvolver.cpp:87-148).  ir[c] points to ir_len[c]
 * float32 taps of channel c (host memory, copied during the call).  Same semantics as the
 * reference: trailing taps with |h| < 1e-6 are trimmed, block sizes are rounded up to a power
 * of two, an empty IR is legal (process() then writes zeros), block size 0 -> B200CONV_EINVAL. */
int b200conv_init_uniform(b200conv_t* h, size_t block, const float* const* ir, const size_t* ir_len);
int b200conv_init_twostage(b200conv_t* h, size_t head_block, size_t tail_block,
                           const float* const* ir, const size_t* ir_len);
/* Non-uniform schedule (beyond the reference): stage s uses block size blocks[s] for the taps
 * [offsets[s], offsets[s+1]) (offsets[0] = 0, last stage runs to the end of the IR).  Stage 0
 * is the zero-latency head; for s >= 1 offsets[s] must be a multiple of blocks[s] and >= blocks[s]. */
int b200conv_init_stages(b200conv_t* h, int n_stages, const size_t* blocks, const size_t* offsets,
                         const float* const* ir, const size_t* ir_len);

/* Streaming convolution (replaces FFTConvolver::process FFTConvolver.cpp:155-212 and
 * TwoStageFFTConvolver::process TwoStageFFTConvolver.cpp:151-233): in[c] / out[c] are HOST
 * pointers to `len` float32 samples per channel; any len >= 0, zero added latency, output is
 * complete on return.  in/out may not alias (same rule as the reference, SURVEY §8a-2).
 * Long calls are internally cut into block batches and pipelined over PCIe. */
int b200conv_process(b200conv_t* h, const float* const* in, float* const* out, size_t len);

/* Same, with DEVICE-resident buffers: channel c at in_dev + c*in_stride (floats).  Asynchronous
 * on the handle's stream unless sync != 0.  This is the throughput path bench.py times. */
int b200conv_process_device(b200conv_t* h, const float* in_dev, size_t in_stride,
                            float* out_dev, size_t out_stride, size_t len, int sync);

/* Time-slice sharding of an offline / batch call over several GPUs — no collective, no exchange.  Every GPU holds
 * the WHOLE convolver (a handle with the same IR and the same history, shard_count = 1); for one call of `len`
 * samples GPU `slice_rank` of `slice_count` produces only the output blocks [a, b) of its contiguous time slice
 * (ceil(T / slice_count) blocks each) and writes out[c][a*B .. b*B) — the rest of `out` is left untouched for the
 * other GPUs (which are given the same `in` / `out` arrays, e.g. one shared, pinned host buffer, or run in other
 * threads of the same process).  The sum over partitions of FFTConvolver.cpp:179-187 needs the spectra of the P
 * blocks in front of a slice: the GPU uploads and forward-transforms that history (FFT only, no sweep), convolves its
 * slice, then transforms the last P blocks of the call, so that after the call EVERY handle is in the state the
 * whole call would have left (the next call — sliced or not — continues the stream).  Per GPU: T/G + P blocks
 * of H2D and forward FFT, T/G blocks of sweep, inverse FFT and D2H.  Pays off when T/G >> P (batch jobs); for
 * streaming calls and IRs longer than the batch use the partition-range shards below.
 * Needs: uniform (single-stage) handle, no routing, no open block, len a multiple of the block size
 * (else B200CONV_ESTATE, nothing processed). */
int b200conv_process_sliced(b200conv_t* h, const float* const* in, float* const* out, size_t len,
                            int slice_rank, int slice_count);
int b200conv_process_device_sliced(b200conv_t* h, const float* in_dev, size_t in_stride, float* out_dev, size_t out_stride,
                                   size_t len, int slice_rank, int slice_count, int sync);

/* FFTConvolver::clear (FFTConvolver.cpp:80-90) / TwoStageFFTConvolver::clear (:69-84): forget
 * all audio history, keep the IR.  Implemented as a TRUE clear (also mid-block), see DESIGN.md. */
int b200conv_clear(b200conv_t* h);
/* FFTConvolver::reset (FFTConvolver.cpp:56-78): drop the IR and all device memory. */
int b200conv_reset(b200conv_t* h);

/* Introspection --------------------------------------------------------------------------- */
typedef struct b200conv_stage_info {
  size_t block;        /* B_s                                  */
  size_t partitions;   /* P_s (max over channels, post-trim)    */
  size_t tap_offset;   /* first IR tap handled by this stage     */
  size_t p_begin;      /* partition range owned by this shard    */
  size_t p_end;
} b200conv_stage_info;
int    b200conv_num_stages(const b200conv_t* h);
int    b200conv_stage(const b200conv_t* h, int s, b200conv_stage_info* out);
size_t b200conv_ir_len(const b200conv_t* h, int channel);    /* post-trim tap count            */
/* Kernel launches issued by this handle since creation (bench.py's gpu_launches). */
unsigned long long b200conv_launch_count(const b200conv_t* h);
/* Form of the FDL sweep (FFTConvolver.cpp:176-187) the last launch resolved to: 22 / 26 = packed-FMA batched sweep,
 * 40 = tensor-core sweep (tcgen05 kind::tf32, 3xTF32), 100..108 = streaming forms.  For benchmarks and tests. */
int b200conv_last_sweep_variant(const b200conv_t* h);
/* Tuning / A-B switches: "rt" (1 = real-time calls that stay inside the open block run as ONE cluster-kernel launch
 * with zero-copy I/O, 0 = multi-kernel path), "fft512" (1 = register-resident FFT kernels for block size 512),
 * "slice_keep_tail" (default 1; 0 = b200conv_process_sliced does not upload / transform the last P blocks of the call:
 * the handle then only supports a following sliced call whose slice starts >= P blocks into the call — every rank
 * but 0 of a steady batch job — until the next b200conv_clear), "stream_alternate" (default 1: the streaming sweep
 * walks its partition slices in alternating directions from launch to launch, see kernels_stream.cuh), "tc" (default 1:
 * launch groups of >= 4096 blocks with <= 961 partitions run the sweep on the tensor cores, kernels_tc.cuh; 0 = always
 * the packed-FMA sweep). */
int    b200conv_set_option(b200conv_t* h, const char* name, int value);
/* Device time (ms) spent in the dominant CMAC kernel / all kernels during the last
 * b200conv_process_device call, measured with CUDA events on the handle's stream
 * (enabled by b200conv_set_timing(h, 1); adds two event records per kernel). */
int    b200conv_set_timing(b200conv_t* h, int enable);
int    b200conv_last_timing(const b200conv_t* h, float* cmac_ms, float* fft_ms, float* ifft_ms,
                            int* cmac_launches);
void*  b200conv_stream(const b200conv_t* h);                  /* cudaStream_t of the head path  */

/* Multi-GPU partition-range sharding (SURVEY §8e): with shard_count > 1 every handle computes
 * the partial spectrum sum over its own partition range; between the CMAC sweep and the
 * inverse FFT the engine calls `reduce(user, dev_ptr, n_floats, stream)` which must sum the
 * buffer over all shards into shard 0 (ncclReduce on that stream).  Only shard 0 produces output;
 * the other shards do not write their `out` buffers. */
typedef int (*b200conv_reduce_fn)(void* user, float* dev_buf, size_t n_floats, void* cuda_stream);
int b200conv_set_reduce(b200conv_t* h, b200conv_reduce_fn fn, void* user);

/* Optional I/O routing of a multi-convolver handle (SURVEY 8f-1: StereoConvolver as ONE call incl.
 * the true-stereo mixdown of src/PluginProcessor.cpp:1833-1838).  Convolver c reads input buffer
 * in_map[c] (0 <= in_map[c] < n_in) and output o = sum_c mix[o*C + c] * y_c, computed on the device.
 * Afterwards b200conv_process / b200conv_process_device take n_in input and n_out output buffers
 * (e.g. quad reverb: in = {L, R}, convolvers {LL, RR, LR, RL} <- {0, 1, 0, 1}, out L = LL + RL,
 * out R = RR + LR: 2 buffers each way over PCIe instead of 4).  n_in = 0 removes the routing.
 * Limits: C <= 8, n_in <= 8, n_out <= 8; not combinable with the slot exchange. */
int b200conv_set_routing(b200conv_t* h, int n_in, const int* in_map, int n_out, const float* mix);

/* The per-sample chain REEV-R runs on the host around the convolver (SURVEY 8f-4 and the rest of 8f-1), on the device:
 *   send: dry * ysend -> low cut (HP) if lowcut_hz > 20 -> high cut (LP) if highcut_hz < 20000 -> predelay ring
 *         (src/PluginProcessor.cpp:1639-1653, 1766-1790; filters = src/dsp/Filter.cpp state-variable sections, slope
 *         0/1/2 = 6/12/24 dB, coefficients as Filter::init / getCoeff compute them);
 *   convolvers LL, RR[, LR, RL] on the chain's L / R (a C = 2 or C = 4 handle);
 *   wet:  L = LL (+ RL), R = RR (+ LR when true_stereo) ; * yrev ; mid/side width ; out = drygain * dry + wetgain * wet
 *         (src/PluginProcessor.cpp:1832-1876).
 * dry[2] / out[2]: host L, R; ysend / yrev: per-sample send and reverb envelopes (NULL = 1).  One H2D of the dry
 * signal + envelopes and one D2H of the final mix per call, whatever the number of convolvers.
 * b200conv_chain_configure(h, cfg) after the IR is loaded (resets filter states and the delay line; NULL disables). */
typedef struct b200conv_chain_config {
  double srate;
  float lowcut_hz;  int lowcut_slope;
  float highcut_hz; int highcut_slope;
  int predelay;                 /* samples */
  float width, drygain, wetgain;
  int true_stereo;              /* quad handles: add RL to the left and LR to the right */
} b200conv_chain_config;
int b200conv_chain_configure(b200conv_t* h, const b200conv_chain_config* cfg);
int b200conv_chain_process(b200conv_t* h, const float* const* dry, const float* ysend, const float* yrev,
                           float* const* out, size_t len);

/* IR hot-swap helpers (SURVEY 8f-2; the reference replays a 0.25 s "warmer" ring through the freshly
 * loaded convolver call by call and crossfades two convolvers on the host for 50 ms,
 * src/PluginProcessor.cpp:1695-1750,1800-1830).
 * b200conv_prime: feeds `len` samples of history through the handle in ONE batched call, no output.
 * b200conv_process_xfade: runs both handles on the same input and returns
 *   out[c][i] = (1 - a_i) * old[c][i] + a_i * new[c][i],  a_i = clamp(alpha0 + i*alpha_step, 0, 1),
 *   blended on the device (one D2H).  Both handles: same device, same channel count / routing, unsharded. */
int b200conv_prime(b200conv_t* h, const float* const* in, size_t len);
int b200conv_process_xfade(b200conv_t* h_old, b200conv_t* h_new, const float* const* in, float* const* out,
                           size_t len, float alpha0, float alpha_step);

/* Fused multi-GPU path ("slot exchange", uniform single-stage handles with shard_count > 1):
 * the sweep kernel's epilogue stores each partial spectrum row straight into the exchange buffer of
 * the GPU that owns the row's time slice (peer memory over NVLink), a flag barrier follows, every
 * GPU runs the inverse FFT on its own slice (summing the shard_count partial slots while loading)
 * and writes the audio directly into shard 0's output exchange buffer.  No NCCL call on the data
 * path.  Set-up: every shard exports a blob, the caller all-gathers the blobs (rank order) and
 * every shard imports the concatenation.  mode 0 = CUDA IPC handles (one process per GPU),
 * mode 1 = raw pointers (all shards in one process on one device; tests). */
size_t b200conv_p2p_blob_size(const b200conv_t* h);
int    b200conv_p2p_export(b200conv_t* h, void* blob, int mode);
int    b200conv_p2p_import(b200conv_t* h, const void* all_blobs /* shard_count * blob_size bytes */);
/* Back to the reduce-hook path (e.g. when the import failed on some other shard: all shards must agree). */
int    b200conv_p2p_detach(b200conv_t* h);
/* Host-pointer calls (b200conv_process) on a slot-exchange handle: with the input broadcast enabled only
 * shard 0 reads its `in` buffers and crosses PCIe; it stores every launch group into the peers' staging
 * buffers over NVLink (the other shards' `in` arguments are ignored).  Off by default (round 1: implemented and
 * covered by the in-process tests, not yet timed on a multi-GPU box). */
int    b200conv_p2p_set_input_broadcast(b200conv_t* h, int enable);
/* Host-side barrier used instead of the flag kernel by the CPU emulation build (tests only). */
typedef int (*b200conv_barrier_fn)(void* user);
int    b200conv_p2p_set_host_barrier(b200conv_t* h, b200conv_barrier_fn fn, void* user);

/* SURVEY 8f-3 (a "next" row, not part of the hot path): the STFT decay-EQ of the IR shaping,
 * Impulse::applyDecay (src/dsp/Impulse.cpp:602-648), on the device: `ir` (host, n float32 taps) is
 * processed in place; lut = 2049 per-bin decay factors per STFT block (Impulse.cpp:566-590 builds them
 * on the host from the EQ bands); srate as in the reference (sets the early-reflection blocks that are
 * left untouched).  Stand-alone call: no handle, own temporary device buffers. */
int b200conv_ir_decay_eq(int device, float* ir, size_t n, const double* lut, double srate);

/* SURVEY 8f-3, the pipeline: the device-resident subset of Impulse::recalcImpulse (src/dsp/Impulse.cpp:297-360) in the
 * reference's order — auto gain (:313-320, :703-720), reverse (:322-330), trim (:437-470), gain (:472-486), decay EQ
 * (:602-648), clip (:488-501), attack / decay envelope (:651-680) — on the raw taps of all 2 / 4 channels with ONE upload.
 * (Resampling, stretch and the parametric EQ stay on the host.)
 *   b200conv_ir_shape            shaped taps back to the host (out[c] needs room for n floats, *out_len taps written);
 *   b200conv_init_*_shaped       shape on the device and build the partition spectra straight from the device-resident
 *                                taps — the IR never returns to the host between shaping and FFTConvolver::init. */
typedef struct b200conv_ir_shape_params {
  int autogain, reverse;
  float trim_left, trim_right;      /* fractions of the length removed at either end */
  float gain;
  const double* decay_lut;          /* 2049 per-bin decay factors (Impulse.cpp:566-590), NULL = no decay EQ */
  double srate;
  int clip;
  float attack, decay;              /* fractions of the (trimmed) length */
} b200conv_ir_shape_params;
int b200conv_ir_shape(int device, const float* const* raw, int n_channels, size_t n, const b200conv_ir_shape_params* sp,
                      float* const* out, size_t* out_len);
int b200conv_init_uniform_shaped(b200conv_t* h, size_t block, const float* const* raw, size_t n,
                                 const b200conv_ir_shape_params* sp);
int b200conv_init_twostage_shaped(b200conv_t* h, size_t head_block, size_t tail_block, const float* const* raw, size_t n,
                                  const b200conv_ir_shape_params* sp);

/* Pinned host memory helpers (staging buffers for the e2e path).  register/unregister page-lock memory the caller
 * owns (e.g. a shared-memory region several per-GPU processes write their output slices into). */
void* b200conv_alloc_host(size_t bytes);
void  b200conv_free_host(void* p);
int   b200conv_register_host(void* p, size_t bytes);
int   b200conv_unregister_host(void* p);

/* Version / build info string ("b200conv x.y sm_100a ..."). */
const char* b200conv_version(void);

#ifdef __cplusplus
}
#endif
#endif /* B200CONV_H */
