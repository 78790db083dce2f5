"""CPU model of the rounding of the FFT sweep along the block axis (reevr_b200/csrc/kernels_tfft.cuh) against the FP32
direct sum of the FFMA sweep, at the metric shape per bin: P = 938 partitions, 6318 output blocks of one channel.

  * reference: float64 linear convolution of the bin's time line with its partition line;
  * "direct fp32": the sum over p in p order, every product and add rounded to float32 (the FFMA sweep's order);
  * "fft N": overlap-save with complex64 transforms of length N (Q = P - 1 history rows per segment), the filter spectra
    computed in float64 and stored as complex64 with 1/N folded in (k_tfft_build_h computes them with the complex64
    transform itself, which adds one more transform's rounding to the filter side).

Errors are max |y - ref| over the peak |ref|, the engine's parity measure.  Run: python tools/tfft_accuracy_model.py
"""
import numpy as np
import scipy.fft as sfft


def line(rng, n):
    return (rng.random(n) - 0.5 + 1j * (rng.random(n) - 0.5)).astype(np.complex64)


def direct_fp32(h, x, T):
    P = h.size
    xp = np.concatenate([np.zeros(P - 1, np.complex64), x])
    acc = np.zeros(T, np.complex64)
    for p in range(P):
        acc = (acc + h[p] * xp[P - 1 - p:P - 1 - p + T]).astype(np.complex64)
    return acc


def fft_overlap_save(h, x, T, N):
    P = h.size
    Q, Lo = P - 1, N - (P - 1)
    Hf = (np.fft.fft(h.astype(np.complex128), N) / N).astype(np.complex64)
    xp = np.concatenate([np.zeros(Q, np.complex64), x, np.zeros(N, np.complex64)])
    y = np.zeros(T, np.complex64)
    for s in range(-(-T // Lo)):
        seg = xp[s * Lo:s * Lo + N]
        z = sfft.fft(seg) * Hf                    # scipy keeps complex64 in single precision
        out = sfft.ifft(z, norm="forward")       # unscaled inverse: 1/N is in Hf
        n = min(Lo, T - s * Lo)
        y[s * Lo:s * Lo + n] = out[Q:Q + n]
    return y


def main(P=938, T=6318, seed=1):
    rng = np.random.default_rng(seed)
    h, x = line(rng, P), line(rng, T)
    ref = np.convolve(x.astype(np.complex128), h.astype(np.complex128))[:T]
    peak = np.max(np.abs(ref))

    def err(y):
        return float(np.max(np.abs(y.astype(np.complex128) - ref)) / peak)
    print(f"P = {P}, {T} output blocks, errors relative to the peak output")
    print(f"  direct fp32 (p order)  {err(direct_fp32(h, x, T)):.2e}")
    for N in (2048, 4096):
        print(f"  fft N = {N:<5}          {err(fft_overlap_save(h, x, T, N)):.2e}")


if __name__ == "__main__":
    main()
