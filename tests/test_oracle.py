"""Pins the CPU oracle (oracle/partconv_oracle.c) — runs without a GPU.

1. the reference's own 58 known-answer cases (naive-convolution truth, reference tolerance);
2. the unmodified reference's output for the same cases and chunking, tight tolerance
   (tests/golden/reference/ref_selftest_cases.npz, generated from oracle/_ref);
3. the committed golden fixtures (tests/golden/*.npz, generated from oracle/_ref).
"""
import glob
import os

import numpy as np
import pytest

from oracle import oracle as orc
from tests import refcases as rc
from tests.golden import make_golden as mg

GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _peak_err(a, b):
    d = np.max(np.abs(a.astype(np.float64) - b.astype(np.float64)))
    return d / max(np.max(np.abs(b.astype(np.float64))), 1e-30)


def _reference_err(fixture, key, y):
    """peak error of y against the reference's stored sample of the same output, relative to its whole peak"""
    g = np.load(os.path.join(mg.REFERENCE, fixture + ".npz"))
    idx = g[key + "_idx"]
    assert idx[-1] == y.size - 1                   # the stored sample always ends on the last sample
    d = np.max(np.abs(y[idx].astype(np.float64) - g[key + "_out"].astype(np.float64)))
    return d / max(float(g[key + "_peak"]), 1e-30)


@pytest.mark.parametrize("case", rc.UNIFORM_CASES, ids=lambda c: "u-" + "-".join(map(str, c)))
def test_uniform_selftest_cases(case):
    n_in, n_ir = case[:2]
    y = mg.selftest_run("uniform", case, "oracle")
    truth = orc.naive_convolve(rc.ramp(n_in), rc.ramp(n_ir))
    assert rc.reference_selftest_ok(y, truth, n_ir)
    assert _reference_err("ref_selftest_cases", mg.selftest_key("uniform", case), y) <= 1e-6


@pytest.mark.parametrize("case", rc.TWOSTAGE_CASES, ids=lambda c: "t-" + "-".join(map(str, c)))
def test_twostage_selftest_cases(case):
    n_in, n_ir = case[:2]
    y = mg.selftest_run("twostage", case, "oracle")
    truth = orc.naive_convolve(rc.ramp(n_in), rc.ramp(n_ir))
    assert rc.reference_selftest_ok(y, truth, n_ir)
    assert _reference_err("ref_selftest_cases", mg.selftest_key("twostage", case), y) <= 1e-6


def test_error_conventions():
    # FFTConvolver.cpp:97-111,157-161: zero block -> false; empty / sub-threshold IR -> true, zeros out
    c = orc.OracleUniform()
    assert not c.init(0, np.ones(4, np.float32))
    assert c.init(8, np.zeros(0, np.float32))
    assert np.all(c.process(np.ones(5, np.float32)) == 0)
    assert c.init(8, np.full(16, 5e-7, np.float32))
    assert np.all(c.process(np.ones(5, np.float32)) == 0)
    # trailing-tap trim is absolute 1e-6 and changes P (FFTConvolver.cpp:103-106)
    h = np.ones(20, np.float32)
    h[17:] = 9e-7
    assert c.init(8, h) and c.partitions == 3   # 17 taps -> ceil(17/8)
    t = orc.OracleTwoStage()
    assert not t.init(0, 8, h) and not t.init(8, 0, h)
    # non power of two rounds up (FFTConvolver.cpp:113)
    assert c.init(5, h) and c.block == 8


def test_clear_block_aligned_gives_zeros():
    # FFTConvolver.cpp:80-90 — a clear() on a block boundary silences the tail completely
    h = orc.synth_ir(1000)
    x = orc.synth_input(512)
    for conv in (orc.OracleUniform(), orc.OracleTwoStage()):
        if isinstance(conv, orc.OracleTwoStage):
            conv.init(32, 128, h)
        else:
            conv.init(64, h)
        conv.process(x)          # 512 = multiple of every block size involved
        conv.clear()
        y = conv.process(np.zeros(2048, np.float32))
        assert np.all(y == 0)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "*.npz"))),
                         ids=lambda p: os.path.basename(p))
def test_golden_fixture(path):
    from tests.golden.make_golden import run_case
    g = np.load(path, allow_pickle=False)
    spec = {k: (g[k].item() if g[k].ndim == 0 else g[k]) for k in g.files if k != "out"}
    y = run_case(spec, impl="oracle")
    assert y.shape == g["out"].shape
    assert _peak_err(y, g["out"]) <= 1e-6


def test_apply_decay_restatement_properties():
    """Groundwork for SURVEY 8f-3 (IR shaping on the device, a 'next' row): the STFT decay of
    src/dsp/Impulse.cpp:602-648.  Unpinned (Impulse.cpp needs JUCE): checked against an independent float64
    numpy model and through the identity property."""
    sr = 48000.0
    h = orc.synth_ir(30000)
    # (1) unit LUT: windowed overlap-add divided by the summed window reproduces the input
    # (the very first samples are ill-conditioned in the reference itself: the window starts at 0, so sample 0
    #  comes back as 0 and the next few are divided by a tiny window sum, Impulse.cpp:646-648)
    y = orc.apply_decay(h, np.ones(2049), sr)
    assert y[0] == 0.0
    assert np.max(np.abs(y[64:1024] - h[64:1024])) <= 1e-4 * np.max(np.abs(h))
    assert np.max(np.abs(y[1024:] - h[1024:])) <= 2e-6 * np.max(np.abs(h))
    # (2) frequency-dependent decay vs an independent float64 model
    lut = np.linspace(1.0, 0.7, 2049)
    w = orc.decay_window().astype(np.float64)
    N, hop = 4096, 1024
    n = h.size
    out = np.zeros(n)
    norm = np.zeros(n)
    skip = int(np.ceil(100 * sr / (1000.0 * N)))
    nblocks = (n + hop - 1) // hop
    for b in range(nblocks):
        s0 = b * hop
        bs = min(N, n - s0)
        blk = np.zeros(N)
        blk[:bs] = h[s0:s0 + bs].astype(np.float64) * w[:bs]
        X = np.fft.rfft(blk)
        if b > skip:
            g = lut ** (b - skip)
            g[0] = 1.0
            X = X * g
        yb = np.fft.irfft(X, N)
        out[s0:s0 + bs] += yb[:bs]
        norm[s0:s0 + bs] += w[:bs]
    want = np.where(norm > 0, out / np.where(norm > 0, norm, 1), 0.0)
    got = orc.apply_decay(h, lut, sr)
    assert np.max(np.abs(got[64:1024] - want[64:1024])) <= 1e-4 * np.max(np.abs(want))
    assert np.max(np.abs(got[1024:] - want[1024:])) <= 1e-5 * np.max(np.abs(want))
    assert np.sum(got[-8000:] ** 2) < 0.2 * np.sum(h[-8000:] ** 2)      # the tail really decays faster


def test_apply_decay_restatement_pinned_by_the_reference_fft():
    """oc_apply_decay (Impulse::applyDecay restated, own FFT) against the same STFT loop driven through the reference's
    compiled audiofft::AudioFFT (oracle/ref_shim.cpp::ref_stft_decay, stored in tests/golden/reference/ref_apply_decay.npz):
    the (f3) oracle is no longer unpinned."""
    for n in mg.DECAY_LENGTHS:
        h = orc.synth_ir(n)
        for j, lut in enumerate(mg.decay_luts()):
            a = orc.apply_decay(h, lut, 48000.0)
            assert _reference_err("ref_apply_decay", f"n{n}_lut{j}", a) <= 1e-6, (n, j)
