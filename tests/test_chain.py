"""SURVEY 8f-4 + the rest of 8f-1: the send / wet chain of processBlock on the device (b200conv_chain_process) against
its oracle (oracle/chain_oracle.c), which is PINNED by the reference's own Filter.cpp compiled into oracle/_ref (its
outputs are stored in tests/golden/reference/ref_filter.npz)."""
import os

import numpy as np
import pytest

from oracle import oracle as orc
from reevr_b200.convolver import Engine
from tests.backends import lib  # noqa: F401
from tests.golden import make_golden as mg

TOL = 1e-5


def peak_err(y, ref):
    return float(np.max(np.abs(y - ref)) / max(np.max(np.abs(ref)), 1e-30))


def test_filter_restatement_is_bit_identical_to_the_reference_filter():
    g = np.load(os.path.join(mg.REFERENCE, "ref_filter.npz"))
    x = mg.filter_input()
    for i, sr in enumerate(mg.FILTER_RATES):
        for j, fr in enumerate(mg.FILTER_FREQS):
            assert orc.filter_coeff(fr, sr) == g["coeff"][i, j]
            for slope in (0, 1, 2):
                for mode in (0, 1, 2):
                    a = orc.OracleFilter(slope, mode, sr, fr, mg.filter_q(slope)).run(x)
                    assert np.array_equal(a[g["idx"]], g["sample"][i, j, slope, mode]), (sr, fr, slope, mode)
                    assert np.array_equal(mg.sha256_u8(a), g["sha256"][i, j, slope, mode]), (sr, fr, slope, mode)


def _reference_chain(cfg, irs, head, tail, L, R, ysend, yrev, chunks):
    """oracle chain + oracle two-stage convolvers, call by call"""
    ch = orc.OracleChain(cfg["srate"], cfg["lowcut_hz"], cfg["lowcut_slope"], cfg["highcut_hz"], cfg["highcut_slope"],
                         cfg["predelay"], cfg["width"], cfg["drygain"], cfg["wetgain"], delay_size=1 << 16)
    convs = []
    for ir in irs:
        o = orc.OracleTwoStage()
        assert o.init(head, tail, ir)
        convs.append(o)
    outL, outR, pos = [], [], 0
    for k in chunks:
        sl = slice(pos, pos + k)
        a, b = ch.send(L[sl], R[sl], ysend[sl])
        ys = [convs[c].process(a if c % 2 == 0 else b) for c in range(len(irs))]
        quad = len(irs) == 4 and cfg["true_stereo"]
        oL, oR = ch.wet(L[sl], R[sl], ys[0], ys[1], ys[2] if quad else None, ys[3] if quad else None, yrev[sl])
        outL.append(oL)
        outR.append(oR)
        pos += k
    return np.concatenate(outL), np.concatenate(outR)


@pytest.mark.parametrize("quad", [False, True])
@pytest.mark.parametrize("cfgid", [0, 1, 2, 3])
def test_chain_against_oracle(lib, quad, cfgid):
    cfgs = [
        dict(srate=48000.0, lowcut_hz=20.0, lowcut_slope=0, highcut_hz=20000.0, highcut_slope=0, predelay=0,
             width=1.0, drygain=1.0, wetgain=1.0, true_stereo=True),                                   # everything neutral
        dict(srate=48000.0, lowcut_hz=180.0, lowcut_slope=1, highcut_hz=6000.0, highcut_slope=2, predelay=777,
             width=0.4, drygain=0.8, wetgain=0.6, true_stereo=True),
        dict(srate=44100.0, lowcut_hz=60.0, lowcut_slope=2, highcut_hz=12000.0, highcut_slope=0, predelay=50,
             width=1.7, drygain=0.0, wetgain=1.0, true_stereo=False),
        dict(srate=96000.0, lowcut_hz=400.0, lowcut_slope=0, highcut_hz=20000.0, highcut_slope=1, predelay=4000,
             width=0.0, drygain=0.5, wetgain=0.5, true_stereo=True),
    ]
    cfg = cfgs[cfgid]
    nconv = 4 if quad else 2
    head, tail = 128, 512
    irs = [orc.synth_ir(2 * tail + 3 * tail + 31, c) for c in range(nconv)]
    chunks = [128] * 30 + [100, 28] + [128 * 25] + [128] * 10 + [7000]      # real-time calls, a ragged pair, batches
    n = sum(chunks)
    L, R = orc.synth_input(n, 0), orc.synth_input(n, 1)
    rng = np.random.default_rng(9)
    ysend = (0.5 + 0.5 * np.abs(np.sin(np.arange(n) * 1e-3))).astype(np.float32)
    yrev = (0.25 + 0.75 * rng.random(n)).astype(np.float32)
    e = Engine(nconv, lib=lib)
    assert e.init_twostage(head, tail, irs)
    e.chain_configure(**cfg)
    gl, gr, pos = [], [], 0
    for k in chunks:
        a, b = e.chain_process(L[pos:pos + k], R[pos:pos + k], ysend[pos:pos + k], yrev[pos:pos + k])
        gl.append(a)
        gr.append(b)
        pos += k
    gl, gr = np.concatenate(gl), np.concatenate(gr)
    wl, wr = _reference_chain(cfg, irs, head, tail, L, R, ysend, yrev, chunks)
    scale = max(np.max(np.abs(wl)), np.max(np.abs(wr)))
    assert np.max(np.abs(gl - wl)) <= TOL * scale and np.max(np.abs(gr - wr)) <= TOL * scale


def test_chain_clear_and_reconfigure(lib):
    irs = [orc.synth_ir(3000, c) for c in range(2)]
    e = Engine(2, lib=lib)
    assert e.init_uniform(64, irs)
    cfg = dict(srate=48000.0, lowcut_hz=100.0, lowcut_slope=2, highcut_hz=9000.0, highcut_slope=1, predelay=300,
               width=0.8, drygain=0.3, wetgain=0.9, true_stereo=True)
    e.chain_configure(**cfg)
    L, R = orc.synth_input(64 * 50, 0), orc.synth_input(64 * 50, 1)
    first = e.chain_process(L, R)
    e.clear()                                    # convolver history, filter states and delay line all start over
    again = e.chain_process(L, R)
    assert np.array_equal(first[0], again[0]) and np.array_equal(first[1], again[1])
    from reevr_b200.convolver import B200ConvError
    with pytest.raises(B200ConvError):
        e.set_routing([0, 1], [[1, 0], [0, 1]])


# ---- SURVEY 8f-3: IR shaping pipeline on the device -------------------------------------------------------------
def _shape_cases():
    return [
        dict(autogain=True, reverse=False, trim_left=0.0, trim_right=0.0, gain=1.0, lut=None, clip=True, attack=0.0, decay=0.0),
        dict(autogain=True, reverse=True, trim_left=0.1, trim_right=0.05, gain=40.0, lut=np.linspace(1.0, 0.8, 2049), srate=48000.0,
             clip=True, attack=0.02, decay=0.3),
        dict(autogain=False, reverse=False, trim_left=0.0, trim_right=0.25, gain=0.5, lut=np.linspace(0.9, 1.04, 2049), srate=44100.0,
             clip=False, attack=0.0, decay=0.5),
    ]


@pytest.mark.parametrize("case", [0, 1, 2])
@pytest.mark.parametrize("nch", [2, 4])
def test_ir_shape_pipeline_against_oracle(lib, case, nch):
    from reevr_b200.convolver import ir_shape
    shape = _shape_cases()[case]
    raws = [orc.synth_ir(21000, c) * (3.0 if c == 1 else 1.0) for c in range(nch)]
    want = orc.ir_shape(raws, **shape)
    got = ir_shape(raws, lib=lib, **shape)
    assert got[0].size == want[0].size
    peak = max(np.max(np.abs(w)) for w in want)
    for c in range(nch):
        # the first STFT hop is ill-conditioned in the reference itself when the decay EQ is on (window starts at 0)
        lo = 1024 if shape["lut"] is not None else 0
        assert np.max(np.abs(got[c][lo:] - want[c][lo:])) <= 1e-5 * peak, (c, case)


def test_shaped_init_equals_shape_then_init(lib):
    """b200conv_init_twostage_shaped (taps never leave the device) == shaping with the oracle, then a plain init"""
    shape = _shape_cases()[1]
    raws = [orc.synth_ir(30000, c) for c in range(2)]
    shaped = orc.ir_shape(raws, **shape)
    x = [orc.synth_input(128 * 60, c) for c in range(2)]
    e = Engine(2, lib=lib)
    assert e.init_twostage_shaped(128, 1024, raws, **shape)
    ys = e.process(x)
    for c in range(2):
        o = orc.OracleTwoStage()
        assert o.init(128, 1024, shaped[c])
        ref = o.process(x[c])
        assert np.max(np.abs(ys[c] - ref)) <= 2e-5 * np.max(np.abs(ref))
    assert abs(e.ir_len(0) - len(orc.ir_shape(raws, **shape)[0])) <= 64      # post-trim length (1e-6 rule) close to the oracle's
