"""Standalone timing of the FFT sweep along the block axis (reevr_b200/csrc/kernels_tfft.cuh, cmac_variant 50..52).

For every candidate transform length N and bin group G it runs the engine with the variant forced, at the metric shape
(stereo, 480 000-tap IR, B = 512, P = 938, T = 112 608 blocks) and at the shape of one of eight time slices
(T = 14 076), and prints:
  * build_h + first sweep, and the steady sweep, from the engine's CUDA events around the sweep launch (median);
  * the sweep's HBM bytes and FP32 flops from the shapes (model() below), the share of the HBM and FP32 peaks and which
    of the two bounds the kernel;
  * the peak error of the sweep output stream against the FFMA sweep (variant 22) on the same input.
The FFMA and tensor-core sweeps (22, 40) are timed the same way for reference.

Run on the GPU:  python tools/tfft_sweep_bench.py [--reps 10] [--out profiles/r03_tfft_sweep.txt]
"""
import argparse
import math
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

VARIANTS = {50: (4096, 4), 51: (2048, 4), 52: (2048, 8)}


def qmax(N):
    """longest history a length-N transform carries (kernels_tfft.cuh tfft_qmax)"""
    return N - N // 4


def model(N, G, C, B, P, T):
    """geometry (kernels_tfft.cuh tfft_geom), HBM bytes and FP32 flops of one sweep launch of T blocks"""
    Q = P - 1
    Lo = N - Q
    nseg = -(-T // Lo)
    lines = C * B
    tiles = lines // G * nseg
    x_bytes = lines * nseg * N * 8          # X rows read, including the Q overlap rows of every segment
    y_bytes = lines * T * 8
    hf_bytes = lines * N * 8                # filter spectra: read once per tile, L2 resident (C*B*N*8 bytes)
    fft = 5.0 * N * math.log2(N)            # flops of one complex radix-2-equivalent transform
    flops = lines * nseg * (2 * fft + 6.0 * N)
    return dict(N=N, G=G, Q=Q, Lo=Lo, nseg=nseg, tiles=tiles, x_bytes=x_bytes, y_bytes=y_bytes, hf_bytes=hf_bytes,
                hbm_bytes=x_bytes + y_bytes, flops=flops)


def peaks():
    """(HBM GB/s, FP32 TFLOP/s): the measured HBM rate of MEASURED_PEAKS.json if present, FP32 from the SM clock"""
    import json
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    hbm, mhz = 6650.0, 1965.0
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        hbm, mhz = float(d["hbm_gbs"]), float(d.get("sm_max_mhz", mhz))
    return hbm, 148 * 128 * 2 * mhz * 1e6 / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    from reevr_b200.convolver import Engine
    from reevr_b200.synth import synth_ir

    C, B = 2, 512
    irs = [synth_ir(480000, c) for c in range(C)]
    P = -(-max(len(h) for h in irs) // B)
    hbm, fp32 = peaks()
    lines = []

    def emit(s=""):
        print(s, flush=True)
        lines.append(s)

    emit(f"# {torch.cuda.get_device_name(0)}; HBM peak {hbm:.0f} GB/s, FP32 peak {fp32:.1f} TFLOP/s; C={C} B={B} P={P}")
    for T in (112608, 14076):
        n = T * B
        g = torch.Generator(device="cpu").manual_seed(7)
        x = (torch.rand((C, n), generator=g) - 0.5).cuda()
        outs = {}
        emit(f"\n## T = {T} blocks")
        emit("variant  N     G  Q    Lo    nseg  first_ms  sweep_ms  HBM_GB  GFLOP   HBM_frac  FP32_frac  bound  err_vs_22")
        for v in (22, 40, 50, 51, 52):
            e = Engine(C, max_batch_blocks=T + 1, cmac_variant=v)
            assert e.init_uniform(B, irs)
            y = torch.zeros_like(x)
            e.set_timing(True)
            e.process_device(x.data_ptr(), n, y.data_ptr(), n, n, sync=True)
            first = e.last_timing()["cmac_ms"]
            ts = []
            for _ in range(args.reps):
                e.clear()
                e.process_device(x.data_ptr(), n, y.data_ptr(), n, n, sync=True)
                ts.append(e.last_timing()["cmac_ms"])
            e.close()
            outs[v] = y.double()
            ms = float(np.median(ts))
            err = float(((outs[v] - outs[22]).abs().max() / outs[22].abs().max()).item())
            if v in VARIANTS:
                m = model(*VARIANTS[v], C, B, P, T)
                fh = m["hbm_bytes"] / (ms * 1e-3) / 1e9 / hbm
                ff = m["flops"] / (ms * 1e-3) / 1e12 / fp32
                emit(f"{v:<8} {m['N']:<5} {m['G']:<2} {m['Q']:<4} {m['Lo']:<5} {m['nseg']:<5} {first:<9.3f} {ms:<9.3f} "
                     f"{m['hbm_bytes'] / 1e9:<7.3f} {m['flops'] / 1e9:<7.1f} {fh:<9.3f} {ff:<10.3f} "
                     f"{'HBM' if fh >= ff else 'FP32':<6} {err:.2e}")
            else:
                emit(f"{v:<8} {'-':<5} {'-':<2} {'-':<4} {'-':<5} {'-':<5} {first:<9.3f} {ms:<9.3f} {'-':<7} {'-':<7} "
                     f"{'-':<9} {'-':<10} {'-':<6} {err:.2e}")
        del x, outs
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
