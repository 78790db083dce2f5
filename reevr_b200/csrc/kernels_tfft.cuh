// kernels_tfft.cuh — batched sweep as an FFT convolution along the block axis (cmac_variant 50..52).
//
// Per bin k and channel the sweep Y[t][k] = sum_{p<P} H[p][k] X[t-p][k] is a linear convolution along the
// block index t with a P-tap filter.  It is evaluated here by overlap-save with a length-N complex FFT along t:
//
//   tile = (channel c, G consecutive bins k0 .. k0+G-1, output segment s of Lo = N - Q blocks), Q = P - 1
//   in[n]  = X[xrow0 + s*Lo - Q + n][k]          n in [0, N)    rows below xlo or from xhi on read as zero
//   out    = IFFT_N( FFT_N(in) .* Hf[c][k] )     Hf = FFT_N(H[0..P-1][k], zero padded) / N  (k_tfft_build_h)
//   Y[yrow0 + s*Lo + n - Q][k] = out[n]          n in [Q, N)    (free of circular wrap because Q >= P - 1)
//
// Entry 0 of a spectrum row packs two real lines (DC, Nyquist).  Its time line z = x_DC + i*x_Ny is transformed
// like any other bin, and so is its filter line h_DC + i*h_Ny; the product step (tfft_apply) separates the two
// real-sequence spectra of both with the (f, N-f) symmetry and recombines W = A*H_DC + i*B*H_Ny, so the real and
// imaginary parts never mix.
//
// Shared memory holds the G time lines of the tile ([G][N + kTfftPad] float2, swizzled with swz() inside each line).
// The FFT passes are the Stockham passes of kernels.cuh (stockham_butterfly, twiddle layout tw_pass_offset(N, p),
// table built in double on the host), run in place: every thread reads its butterflies' inputs into registers,
// the CTA synchronises, every thread stores its outputs.  NT = G*N/32 threads, so a thread holds 32 values per pass.
#pragma once

#include "kernels.cuh"

namespace pc {

constexpr int kTfftPad = 4;           // float2 between the G lines: the two bins of a 16-byte row load hit different banks

constexpr PC_HD int tfft_threads(int N, int G) { return G * N / 32; }
constexpr PC_HD size_t tfft_smem_bytes(int N, int G) { return (size_t)G * (size_t)(N + kTfftPad) * 8u; }
// longest history a length-N transform carries: at least a quarter of every transform is output
constexpr PC_HD int tfft_qmax(int N) { return N - N / 4; }

struct TfftGeom { int Q, Lo, nseg; };

// P = partition rows of the sweep (>= 1), nblocks = output blocks of the launch group
PC_HD TfftGeom tfft_geom(int N, int P, int nblocks) {
  TfftGeom g;
  g.Q = P - 1;
  g.Lo = N - g.Q;
  g.nseg = (nblocks + g.Lo - 1) / g.Lo;
  return g;
}

struct TfftParams {
  const float2* X; long long x_cstride;
  long long xrow0;           // X row of output block 0 at partition 0
  long long xlo, xhi;        // rows outside [xlo, xhi) read as zero
  const float2* Hf;          // [C][B][N] filter spectra (1/N folded in)
  float2* Y; long long y_cstride, y_rstride, yrow0;
  const float2* tw;          // twiddle table of the length-N transform (kernels.cuh layout)
  int B, nblocks, Q, Lo, nseg;
};

struct TfftBuildParams {
  const float2* H; long long h_cstride;   // [C][Prows][B], partition rows [0, P) used
  float2* Hf;                             // [C][B][N]
  const float2* tw;
  int B, P;
};

// tile index -> (channel, bin group, segment); segments vary fastest so that concurrent CTAs share the Q
// overlap rows of neighbouring segments in L2
PC_HD void tfft_tile(int tile, int nseg, int ngroups, int& c, int& grp, int& seg) {
  seg = tile % nseg;
  const int cg = tile / nseg;
  grp = cg % ngroups;
  c = cg / ngroups;
}

// output store of a pass run in place: the butterfly's outputs (issued in order m = 0 .. R-1, offset m*p)
// go to registers until the whole CTA has read its inputs
struct RegOut {
  float2* r; int p;
  PC_HD int prep(int base) const { return base; }
  PC_HD void put(int, int off, float2 v) const { r[off / p] = v; }
};

PC_HD void tfft_pass_write(float2* line, int p, int R, int i, const float2* v) {
  const int k = i & (p - 1);
  const int j = (i - k) * R + k;
  for (int m = 0; m < R; ++m) line[swz(j + m * p)] = v[m];
}

// load phase, element e = (row n, bin pair gp): two adjacent bins of one X row (16 bytes)
template <int N, int G>
PC_HD void tfft_load_pair(const TfftParams& P, int c, int grp, int seg, int e, float2* buf) {
  const int n = e / (G / 2), g = 2 * (e % (G / 2));
  const long long row = P.xrow0 + (long long)seg * P.Lo - P.Q + n;
  float4c v;
  if (row >= P.xlo && row < P.xhi) v = ld_pair(P.X + (long long)c * P.x_cstride + row * P.B + grp * G + g);
  else v.a = v.b = make_float2(0.0f, 0.0f);
  buf[g * (N + kTfftPad) + swz(n)] = v.a;
  buf[(g + 1) * (N + kTfftPad) + swz(n)] = v.b;
}

PC_HD void st_pair(float2* p, float2 a, float2 b) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<float4*>(p) = make_float4(a.x, a.y, b.x, b.y);
#else
  p[0] = a; p[1] = b;
#endif
}

// store phase, element e = (output row n = Q + e / (G/2), bin pair)
template <int N, int G>
PC_HD void tfft_store_pair(const TfftParams& P, int c, int grp, int seg, int e, const float2* buf) {
  const int n = P.Q + e / (G / 2), g = 2 * (e % (G / 2));
  const long long t = (long long)seg * P.Lo + (n - P.Q);
  if (n >= N || t >= P.nblocks) return;
  st_pair(P.Y + (long long)c * P.y_cstride + (P.yrow0 + t) * P.y_rstride + grp * G + g,
          buf[g * (N + kTfftPad) + swz(n)], buf[(g + 1) * (N + kTfftPad) + swz(n)]);
}

// product with the filter spectrum, element e = (bin g, frequency pair f / N-f), f in [0, N/2]
template <int N, int G>
PC_HD void tfft_apply(const TfftParams& P, int c, int grp, int e, float2* buf) {
  const int g = e / (N / 2 + 1), f = e % (N / 2 + 1), fm = (N - f) & (N - 1);
  const int k = grp * G + g;
  float2* line = buf + g * (N + kTfftPad);
  const float2* hf = P.Hf + ((long long)c * P.B + k) * N;
  const float2 zf = line[swz(f)], zm = line[swz(fm)];
  const float2 hff = hf[f], hfm = hf[fm];
  if (k != 0) {
    line[swz(f)] = c_mul(zf, hff);
    if (fm != f) line[swz(fm)] = c_mul(zm, hfm);
    return;
  }
  // (DC, Nyquist): A / B = spectra of the real lines x_DC / x_Ny, Hd / Hn those of h_DC / h_Ny
  const float2 A = make_float2(0.5f * (zf.x + zm.x), 0.5f * (zf.y - zm.y));
  const float2 Bn = make_float2(0.5f * (zf.y + zm.y), -0.5f * (zf.x - zm.x));
  const float2 Hd = make_float2(0.5f * (hff.x + hfm.x), 0.5f * (hff.y - hfm.y));
  const float2 Hn = make_float2(0.5f * (hff.y + hfm.y), -0.5f * (hff.x - hfm.x));
  const float2 a = c_mul(A, Hd), b = c_mul(Bn, Hn);                       // W[f] = a + i*b
  const float2 am = c_mul(c_conj(A), c_conj(Hd)), bm = c_mul(c_conj(Bn), c_conj(Hn));
  line[swz(f)] = make_float2(a.x - b.y, a.y + b.x);
  line[swz(fm)] = make_float2(am.x - bm.y, am.y + bm.x);
}

// build phase: element e = (partition row n, bin g) of the zero-padded filter line
template <int N, int G>
PC_HD void tfft_build_load(const TfftBuildParams& P, int c, int grp, int e, float2* buf) {
  const int n = e / G, g = e % G;
  buf[g * (N + kTfftPad) + swz(n)] =
      n < P.P ? P.H[(long long)c * P.h_cstride + (long long)n * P.B + grp * G + g] : make_float2(0.0f, 0.0f);
}

template <int N, int G>
PC_HD void tfft_build_store(const TfftBuildParams& P, int c, int grp, int e, const float2* buf) {
  const int g = e / N, f = e % N;
  const float2 v = buf[g * (N + kTfftPad) + swz(f)];
  const float s = 1.0f / (float)N;
  P.Hf[((long long)c * P.B + grp * G + g) * N + f] = make_float2(v.x * s, v.y * s);
}

#if defined(__CUDACC__)
// all passes of one length-N transform of the G lines, in place
template <bool INV, int N, int G, int p>
PC_D void tfft_passes(float2* buf, const float2* __restrict__ tw) {
  if constexpr (p < N) {
    constexpr int R = pass_radix(N, p);
    constexpr int NT = tfft_threads(N, G);
    constexpr int NB = G * (N / R) / NT;       // butterflies per thread
    float2 v[NB][8];
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int b = threadIdx.x + j * NT, g = b / (N / R), i = b % (N / R);
      stockham_butterfly<INV>(SmemIn{buf + g * (N + kTfftPad)}, RegOut{v[j], p}, tw + tw_pass_offset(N, p), N, p, R, i);
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < NB; ++j) {
      const int b = threadIdx.x + j * NT, g = b / (N / R), i = b % (N / R);
      tfft_pass_write(buf + g * (N + kTfftPad), p, R, i, v[j]);
    }
    __syncthreads();
    tfft_passes<INV, N, G, p * R>(buf, tw);
  }
}

template <int N, int G>
__global__ void __launch_bounds__(tfft_threads(N, G), 1) k_tfft_sweep(TfftParams P) {
  extern __shared__ float2 tfft_buf[];
  constexpr int NT = tfft_threads(N, G);
  int c, grp, seg;
  tfft_tile(blockIdx.x, P.nseg, P.B / G, c, grp, seg);
#pragma unroll 8
  for (int e = threadIdx.x; e < N * G / 2; e += NT) tfft_load_pair<N, G>(P, c, grp, seg, e, tfft_buf);
  __syncthreads();
  tfft_passes<false, N, G, 1>(tfft_buf, P.tw);
  for (int e = threadIdx.x; e < G * (N / 2 + 1); e += NT) tfft_apply<N, G>(P, c, grp, e, tfft_buf);
  __syncthreads();
  tfft_passes<true, N, G, 1>(tfft_buf, P.tw);
#pragma unroll 8
  for (int e = threadIdx.x; e < (N - P.Q) * G / 2; e += NT) tfft_store_pair<N, G>(P, c, grp, seg, e, tfft_buf);
}

// grid (B / G, C)
template <int N, int G>
__global__ void __launch_bounds__(tfft_threads(N, G), 1) k_tfft_build_h(TfftBuildParams P) {
  extern __shared__ float2 tfft_buf[];
  constexpr int NT = tfft_threads(N, G);
  for (int e = threadIdx.x; e < N * G; e += NT) tfft_build_load<N, G>(P, blockIdx.y, blockIdx.x, e, tfft_buf);
  __syncthreads();
  tfft_passes<false, N, G, 1>(tfft_buf, P.tw);
  for (int e = threadIdx.x; e < N * G; e += NT) tfft_build_store<N, G>(P, blockIdx.y, blockIdx.x, e, tfft_buf);
}
#endif  // __CUDACC__

#if !defined(__CUDACC__)
// CPU emulation (tests/emu): the same phases, threads as loops, each in-place pass as "all threads read, then all
// threads write"
template <bool INV, int N, int G>
inline void emu_tfft_transform(float2* buf, const float2* tw, float2* regs /*[G*N]*/) {
  for (int p = 1; p < N;) {
    const int R = pass_radix(N, p);
    for (int b = 0; b < G * (N / R); ++b) {
      const int g = b / (N / R), i = b % (N / R);
      stockham_butterfly<INV>(SmemIn{buf + g * (N + kTfftPad)}, RegOut{regs + (long long)b * R, p}, tw + tw_pass_offset(N, p), N, p, R, i);
    }
    for (int b = 0; b < G * (N / R); ++b) {
      const int g = b / (N / R), i = b % (N / R);
      tfft_pass_write(buf + g * (N + kTfftPad), p, R, i, regs + (long long)b * R);
    }
    p *= R;
  }
}

template <int N, int G>
inline void emu_tfft_sweep(int C, const TfftParams& P) {
  float2* buf = new float2[tfft_smem_bytes(N, G) / 8];
  float2* regs = new float2[(size_t)G * N];
  const int ngroups = P.B / G;
  for (int tile = 0; tile < C * ngroups * P.nseg; ++tile) {
    int c, grp, seg;
    tfft_tile(tile, P.nseg, ngroups, c, grp, seg);
    for (int e = 0; e < N * G / 2; ++e) tfft_load_pair<N, G>(P, c, grp, seg, e, buf);
    emu_tfft_transform<false, N, G>(buf, P.tw, regs);
    for (int e = 0; e < G * (N / 2 + 1); ++e) tfft_apply<N, G>(P, c, grp, e, buf);
    emu_tfft_transform<true, N, G>(buf, P.tw, regs);
    for (int e = 0; e < (N - P.Q) * G / 2; ++e) tfft_store_pair<N, G>(P, c, grp, seg, e, buf);
  }
  delete[] buf; delete[] regs;
}

template <int N, int G>
inline void emu_tfft_build_h(int C, const TfftBuildParams& P) {
  float2* buf = new float2[tfft_smem_bytes(N, G) / 8];
  float2* regs = new float2[(size_t)G * N];
  for (int c = 0; c < C; ++c)
    for (int grp = 0; grp < P.B / G; ++grp) {
      for (int e = 0; e < N * G; ++e) tfft_build_load<N, G>(P, c, grp, e, buf);
      emu_tfft_transform<false, N, G>(buf, P.tw, regs);
      for (int e = 0; e < N * G; ++e) tfft_build_store<N, G>(P, c, grp, e, buf);
    }
  delete[] buf; delete[] regs;
}
#endif  // !__CUDACC__

}  // namespace pc
