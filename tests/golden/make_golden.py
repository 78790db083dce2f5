"""Generates tests/golden/*.npz from the UNMODIFIED reference (oracle/_ref).

Run where oracle/_ref can be built (the original project's sources, see oracle/Makefile):
    python -m tests.golden.make_golden
Each fixture stores the case parameters, a checksum of the regenerated inputs and the
reference output `out`; `run_case` re-creates the inputs and drives any implementation that
offers the reference surface (init/process/clear), so the same function checks the C oracle
(tests/test_oracle.py) and the CUDA path (tests/test_gpu_parity.py).

Three more fixtures, under reference/, pin the C restatements in oracle/ to the reference where the
tests used to need the compiled reference at test time:
  ref_selftest_cases.npz   reference output of the 58 self-test cases (tests/refcases.py)
  ref_apply_decay.npz      the STFT decay driven through the reference's own AudioFFT
  ref_filter.npz           the reference Filter: coefficients and the SHA-256 of every output
Long outputs are stored as a sample (`sample_points`) plus the peak of the whole output, so the
tests keep their tolerance relative to the full output's peak.
"""
import hashlib
import os
import sys
import zlib

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE = os.path.join(HERE, "reference")
ROOT = os.path.dirname(os.path.dirname(HERE))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import oracle as orc  # noqa: E402
from tests import refcases as rc  # noqa: E402

# name -> spec.  kind: uniform|twostage; signal: synth|ramp; chunking: fixed n | ragged(seed)
CASES = {
    "uniform_b64_ir1000": dict(kind="uniform", block=64, tail=0, ir_len=1000, n=4096, signal="synth", chunk=64, rag=0),
    "uniform_b64_ir1000_ragged": dict(kind="uniform", block=64, tail=0, ir_len=1000, n=4096, signal="synth", chunk=0, rag=7),
    "uniform_b512_ir48000_cfg1": dict(kind="uniform", block=512, tail=0, ir_len=48000, n=512 * 24, signal="synth", chunk=512, rag=0),
    "uniform_b512_ir480000_metric": dict(kind="uniform", block=512, tail=0, ir_len=480000, n=512 * 16, signal="synth", chunk=512, rag=0),
    "uniform_b100_ramp": dict(kind="uniform", block=100, tail=0, ir_len=321, n=3000, signal="ramp", chunk=0, rag=3),
    "uniform_b1_tiny": dict(kind="uniform", block=1, tail=0, ir_len=5, n=40, signal="synth", chunk=0, rag=11),
    "twostage_h32_t256_ir3000": dict(kind="twostage", block=32, tail=256, ir_len=3000, n=4096, signal="synth", chunk=32, rag=0),
    "twostage_h32_t256_ir3000_ragged": dict(kind="twostage", block=32, tail=256, ir_len=3000, n=4096, signal="synth", chunk=0, rag=5),
    "twostage_h128_t8192_ir240000_cfg2": dict(kind="twostage", block=128, tail=8192, ir_len=240000, n=128 * 160, signal="synth", chunk=128, rag=0),
    "twostage_h64_t128_short_ir": dict(kind="twostage", block=64, tail=128, ir_len=100, n=1000, signal="synth", chunk=0, rag=9),
    "uniform_clear_midstream": dict(kind="uniform", block=64, tail=0, ir_len=1000, n=4096, signal="synth", chunk=64, rag=0, clear_at=2048),
    "twostage_clear_midstream": dict(kind="twostage", block=32, tail=256, ir_len=3000, n=4096, signal="synth", chunk=32, rag=0, clear_at=2048),
}


def _signals(spec):
    n, L = int(spec["n"]), int(spec["ir_len"])
    if str(spec["signal"]) == "ramp":
        return rc.ramp(n), rc.ramp(L)
    return orc.synth_input(n), orc.synth_ir(L)


def _chunks(spec):
    n = int(spec["n"])
    if int(spec["rag"]) == 0:
        c = int(spec["chunk"])
        return [c] * (n // c) + ([n % c] if n % c else [])
    rng = np.random.default_rng(int(spec["rag"]))
    hi = 3 * int(spec["block"]) + 2
    out, done = [], 0
    while done < n:
        k = int(min(n - done, rng.integers(1, hi)))
        out.append(k)
        done += k
    return out


def make_impl(spec, impl):
    kind = str(spec["kind"])
    if impl == "ref":
        return orc.RefUniform() if kind == "uniform" else orc.RefTwoStage()
    if impl == "oracle":
        return orc.OracleUniform() if kind == "uniform" else orc.OracleTwoStage()
    return impl(kind)  # factory supplied by the caller (CUDA path)


def run_case(spec, impl="oracle"):
    x, h = _signals(spec)
    conv = make_impl(spec, impl)
    if str(spec["kind"]) == "uniform":
        assert conv.init(int(spec["block"]), h)
    else:
        assert conv.init(int(spec["block"]), int(spec["tail"]), h)
    if "in_crc" in spec:
        assert zlib.crc32(x.tobytes()) == int(spec["in_crc"]), "synthetic input generator drifted"
        assert zlib.crc32(h.tobytes()) == int(spec["ir_crc"]), "synthetic IR generator drifted"
    clear_at = int(spec.get("clear_at", -1))
    y = np.empty_like(x)
    pos = 0
    for k in _chunks(spec):
        if pos == clear_at:   # block-aligned clear (SURVEY §8a-3)
            conv.clear()
        y[pos:pos + k] = conv.process(x[pos:pos + k])
        pos += k
    return y


def sample_points(n: int, k: int = 256) -> np.ndarray:
    """Indices of the stored sample of an n-sample output: all of them when n <= k, else the first and last k/4 and
    k/2 seeded random ones in between (sorted)."""
    if n <= k:
        return np.arange(n, dtype=np.int32)
    q = k // 4
    mid = np.random.default_rng(n).choice(np.arange(q, n - q), k - 2 * q, replace=False)
    return np.sort(np.concatenate([np.arange(q), mid, np.arange(n - q, n)])).astype(np.int32)


def selftest_key(kind: str, case) -> str:
    return kind[0] + "-" + "-".join(map(str, case))


def selftest_run(kind: str, case, impl: str) -> np.ndarray:
    """One case of the reference self-test (ramps, glibc rand() chunking) through the oracle or the reference."""
    x, h = rc.ramp(case[0]), rc.ramp(case[1])
    total = case[0] + case[1] - 1
    chunks = rc.chunk_schedule(total, case[2], case[3], rc.GlibcRand(1))
    if kind == "uniform":
        conv = orc.RefUniform() if impl == "ref" else orc.OracleUniform()
        assert conv.init(case[4], h)
    else:
        conv = orc.RefTwoStage() if impl == "ref" else orc.OracleTwoStage()
        assert conv.init(case[4], case[5], h)
    return rc.drive(conv, x, total, chunks)


DECAY_LENGTHS = (30000, 5000, 4096, 1025, 100)


def decay_luts():
    return (np.ones(2049), np.linspace(1.0, 0.7, 2049), np.linspace(0.8, 1.05, 2049))


FILTER_RATES = (44100.0, 48000.0, 96000.0)
FILTER_FREQS = (20.0, 55.5, 300.0, 1234.0, 8000.0, 19999.0, 30000.0)


def filter_input() -> np.ndarray:
    return np.random.default_rng(3).standard_normal(6000).astype(np.float32)


def filter_q(slope: int) -> float:
    return 0.0765 if slope == 2 else 0.2929


def sha256_u8(a: np.ndarray) -> np.ndarray:
    return np.frombuffer(hashlib.sha256(np.ascontiguousarray(a).tobytes()).digest(), dtype=np.uint8)


def make_ref_selftest_cases() -> dict:
    out = {}
    for kind, cases in (("uniform", rc.UNIFORM_CASES), ("twostage", rc.TWOSTAGE_CASES)):
        for case in cases:
            y = selftest_run(kind, case, "ref")
            idx = sample_points(y.size)
            k = selftest_key(kind, case)
            out[k + "_idx"], out[k + "_out"], out[k + "_peak"] = idx, y[idx], np.float64(np.max(np.abs(y)))
    return out


def make_ref_apply_decay() -> dict:
    out = {}
    for n in DECAY_LENGTHS:
        h = orc.synth_ir(n)
        for j, lut in enumerate(decay_luts()):
            y = orc.ref_apply_decay(h, lut, 48000.0)
            idx = sample_points(y.size)
            k = f"n{n}_lut{j}"
            out[k + "_idx"], out[k + "_out"], out[k + "_peak"] = idx, y[idx], np.float64(np.max(np.abs(y)))
    return out


def make_ref_filter() -> dict:
    """coeff[rate, freq]; sha256 / sample[rate, freq, slope, mode] of the filtered filter_input()"""
    x = filter_input()
    idx = sample_points(x.size, 64)
    coeff = np.zeros((len(FILTER_RATES), len(FILTER_FREQS)))
    sha = np.zeros((len(FILTER_RATES), len(FILTER_FREQS), 3, 3, 32), np.uint8)
    sample = np.zeros((len(FILTER_RATES), len(FILTER_FREQS), 3, 3, idx.size), np.float32)
    for i, sr in enumerate(FILTER_RATES):
        for j, fr in enumerate(FILTER_FREQS):
            coeff[i, j] = orc.filter_coeff(fr, sr, ref=True)
            for slope in range(3):
                for mode in range(3):
                    y = orc.RefFilter(slope, mode, sr, fr, filter_q(slope)).run(x)
                    sha[i, j, slope, mode] = sha256_u8(y)
                    sample[i, j, slope, mode] = y[idx]
    return dict(coeff=coeff, sha256=sha, idx=idx, sample=sample)


def main():
    assert orc.ref_available() and orc.ref_filter_available(), "needs oracle/_ref (the compiled reference)"
    for name, spec in CASES.items():
        x, h = _signals(spec)
        spec = dict(spec, in_crc=zlib.crc32(x.tobytes()), ir_crc=zlib.crc32(h.tobytes()))
        out = run_case(spec, impl="ref")
        np.savez_compressed(os.path.join(HERE, name + ".npz"), out=out, **spec)
        print(f"{name}: {out.size} samples, peak {np.abs(out).max():.4g}")
    for name, make in (("ref_selftest_cases", make_ref_selftest_cases), ("ref_apply_decay", make_ref_apply_decay),
                       ("ref_filter", make_ref_filter)):
        np.savez_compressed(os.path.join(REFERENCE, name + ".npz"), **make())
        print(f"{name}: written")


if __name__ == "__main__":
    main()
