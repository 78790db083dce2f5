"""FFT form of the batched sweep (reevr_b200/csrc/kernels_tfft.cuh, cmac_variant 50..52): per bin, the sum over
partitions is a linear convolution along the block index, evaluated by overlap-save with a length-N FFT along t.
Checked against the oracle (FFTConvolver.cpp:176-187 restated) at 1e-5 of peak and against the FFMA sweep (variant 22)
at 4e-6, over ragged launch groups, groups shorter than one segment and groups of several segments, the largest
supported partition count, a single partition, the packed (DC, Nyquist) entry, two-stage handles, clear() and
time-sliced calls — on the CPU emulation and on the GPU."""
import numpy as np
import pytest

from oracle import oracle as orc
from reevr_b200.convolver import B200ConvError, Engine
from tests.backends import get_lib, lib  # noqa: F401

TOL = 1e-5
TOL_FFMA = 4e-6


def peak_err(y, ref):
    y = np.asarray(y, np.float64)
    ref = np.asarray(ref, np.float64)
    return float(np.max(np.abs(y - ref)) / max(np.max(np.abs(ref)), 1e-30))


def run(eng, xs, chunks):
    outs = [[] for _ in xs]
    pos = 0
    for k in chunks:
        ys = eng.process([x[pos:pos + k] for x in xs])
        for c, y in enumerate(ys):
            outs[c].append(y)
        pos += k
    return [np.concatenate(o) for o in outs]


# (B, partitions, blocks, C, variant, max_batch_blocks).  3073 = Q_max(4096) + 1 and 1537 = Q_max(2048) + 1 are the
# largest partition counts; max_batch_blocks 512 keeps every N = 4096 group inside one segment, the 4096-block groups
# of the variant 51 / 52 cases span several segments with a ragged last one.
CASES = [(512, 938, 260, 2, 50, 512), (32, 3073, 150, 1, 50, 512), (64, 1, 300, 2, 50, 512), (32, 40, 300, 4, 50, 512),
         (64, 100, 700, 1, 50, 512), (32, 1537, 120, 1, 51, 512), (32, 700, 4700, 1, 51, 4096),
         (64, 300, 4500, 2, 52, 4096)]


@pytest.mark.parametrize("B,nparts,nblocks,C,variant,mbb", CASES)
def test_tfft_sweep_matches_oracle_and_ffma(lib, B, nparts, nblocks, C, variant, mbb):
    irs = [orc.synth_ir(nparts * B - (5 if nparts > 1 else 0), c) for c in range(C)]
    n = nblocks * B + 37
    xs = [orc.synth_input(n, c) for c in range(C)]
    chunks = [n // 3 + 11, B - 11, n - (n // 3 + 11) - (B - 11)]       # ragged launch groups, an open block in between
    ys = {}
    for v in (variant, 22):
        e = Engine(C, cmac_variant=v, max_batch_blocks=mbb, lib=lib)
        assert e.init_uniform(B, irs)
        ys[v] = run(e, xs, chunks)
        assert e.last_sweep_variant() == v
        e.close()
    for c in range(C):
        o = orc.OracleUniform()
        o.init(B, irs[c])
        ref = o.process(xs[c])
        assert peak_err(ys[variant][c], ref) <= TOL
        assert peak_err(ys[variant][c], ys[22][c]) <= TOL_FFMA


def test_tfft_sweep_twostage_handle(lib):
    irs = [orc.synth_ir(60000, c) for c in range(2)]
    n = 128 * 900 + 50
    xs = [orc.synth_input(n, c) for c in range(2)]
    e = Engine(2, cmac_variant=50, max_batch_blocks=400, lib=lib)
    assert e.init_twostage(128, 8192, irs)
    ys = run(e, xs, [n // 2 + 3, n - n // 2 - 3])
    e.close()
    for c in range(2):
        o = orc.OracleTwoStage()
        o.init(128, 8192, irs[c])
        assert peak_err(ys[c], o.process(xs[c])) <= TOL


def test_tfft_sweep_clear_midstream(lib):
    B = 64
    ir = orc.synth_ir(300 * B - 7)
    x = orc.synth_input(500 * B + 13)
    e = Engine(1, cmac_variant=50, max_batch_blocks=512, lib=lib)
    assert e.init_uniform(B, [ir])
    e.process([orc.synth_input(200 * B + 5, 3)])
    e.clear()                                         # the history the sweep reads must be gone
    y = run(e, [x], [x.size // 2, x.size - x.size // 2])[0]
    e.close()
    o = orc.OracleUniform()
    o.init(B, ir)
    assert peak_err(y, o.process(x)) <= TOL


def test_tfft_sweep_time_sliced_calls(lib):
    B, G, C = 64, 3, 2
    irs = [orc.synth_ir(260 * B - 3, c) for c in range(C)]
    calls = [(150 * B, True), (40 * B, False), (301 * B, True), (90 * B, True)]
    n = sum(k for k, _ in calls)
    xs = [orc.synth_input(n, c) for c in range(C)]
    engs = [Engine(C, cmac_variant=50, max_batch_blocks=512, lib=lib) for _ in range(G)]
    for e in engs:
        assert e.init_uniform(B, irs)
    outs = [np.zeros(n, np.float32) for _ in range(C)]
    pos = 0
    for k, sliced in calls:
        seg = [np.ascontiguousarray(x[pos:pos + k]) for x in xs]
        if sliced:
            ys = [np.full(k, np.nan, np.float32) for _ in range(C)]
            for g, e in enumerate(engs):
                e.process_sliced(seg, ys, g, G)
        else:
            ys = [e.process(seg) for e in engs][0]
        for c in range(C):
            outs[c][pos:pos + k] = ys[c]
        pos += k
    for e in engs:
        assert e.last_sweep_variant() == 50
        e.close()
    for c in range(C):
        o = orc.OracleUniform()
        o.init(B, irs[c])
        assert peak_err(outs[c], o.process(xs[c])) <= TOL


def test_tfft_sweep_refuses_what_it_cannot_do(lib):
    B = 32
    irs = [orc.synth_ir(3074 * B, 0)]                   # 3074 partitions: Q = 3073 > Q_max(4096) = 3072
    x = [orc.synth_input(40 * B, 0)]
    for variant in (50, 51, 52):
        e = Engine(1, cmac_variant=variant, lib=lib)
        assert e.init_uniform(B, irs)
        with pytest.raises(B200ConvError):
            e.process(x)
        e.close()
    e = Engine(1, cmac_variant=52, lib=lib)             # B = 4 is not a multiple of the 8-bin group
    assert e.init_uniform(4, [orc.synth_ir(4 * 20, 0)])
    with pytest.raises(B200ConvError):
        e.process([orc.synth_input(4 * 80, 0)])
    e.close()
    e = Engine(1, lib=lib)                               # automatic selection never picks it for that shape
    assert e.init_uniform(B, irs)
    y = e.process(x)[0]
    assert e.last_sweep_variant() != 50
    o = orc.OracleUniform()
    o.init(B, irs[0])
    assert peak_err(y, o.process(x[0])) <= TOL
    e.close()


@pytest.mark.gpu
def test_tfft_sweep_is_the_default_at_the_metric_bin_count():
    """B = 512, P = 300, T = 4608: FFT sweep by default, the tensor-core sweep with "tfft" off, the FFMA sweep with
    both off; all three agree."""
    import torch
    lib_ = get_lib("cuda")
    B, nparts, T = 512, 300, 4608
    irs = [orc.synth_ir(nparts * B - 9, c) for c in range(2)]
    n = T * B
    x = np.stack([orc.synth_input(n, c) for c in range(2)])
    xd = torch.from_numpy(x).cuda()
    res = {}
    for tfft, tc, want in ((1, 1, 50), (0, 1, 40), (0, 0, 22)):
        e = Engine(2, max_batch_blocks=T + 1, lib=lib_)
        assert e.init_uniform(B, irs)
        e.set_option("tfft", tfft)
        e.set_option("tc", tc)
        yd = torch.zeros_like(xd)
        e.process_device(xd.data_ptr(), n, yd.data_ptr(), n, n, sync=True)
        assert e.last_sweep_variant() == want
        res[want] = yd.cpu().numpy()
        e.close()
    for c in range(2):
        assert peak_err(res[50][c], res[22][c]) <= TOL_FFMA
        assert peak_err(res[40][c], res[22][c]) <= TOL_FFMA
    o = orc.OracleUniform()
    o.init(B, irs[0])
    assert peak_err(res[50][0][:400 * B], o.process(x[0][:400 * B])) <= TOL


GEOM_SHIM = r"""
#include "kernels_tfft.cuh"
extern "C" void tfft_geom_c(int N, int P, int nb, int* out) {
  const pc::TfftGeom g = pc::tfft_geom(N, P, nb);
  out[0] = g.Q; out[1] = g.Lo; out[2] = g.nseg; out[3] = pc::tfft_qmax(N); out[4] = pc::tfft_threads(N, 4);
  out[5] = (int)pc::tfft_smem_bytes(N, 4);
}
"""


def test_tool_model_matches_the_kernel_geometry(tmp_path):
    """tools/tfft_sweep_bench.py's bytes / flops model uses the header's segment geometry (CPU only)."""
    import ctypes
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src, so = tmp_path / "shim.cpp", tmp_path / "libtfft_geom.so"
    src.write_text(GEOM_SHIM)
    cmd = ["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-I", os.path.join(root, "reevr_b200", "csrc"), str(src), "-o", str(so)]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    lib_ = ctypes.CDLL(str(so))
    sys.path.insert(0, os.path.join(root, "tools"))
    import tfft_sweep_bench as tool
    for (N, G) in tool.VARIANTS.values():
        for P, T in ((938, 112608), (938, 14076), (1, 1), (1, N), (1, N + 1), (tool.qmax(N) + 1, 5000), (300, 4500)):
            buf = (ctypes.c_int * 6)()
            lib_.tfft_geom_c(N, P, T, buf)
            m = tool.model(N, G, 2, 512, P, T)
            assert (m["Q"], m["Lo"], m["nseg"]) == (buf[0], buf[1], buf[2])
            assert tool.qmax(N) == buf[3]
            assert m["nseg"] * m["Lo"] >= T > (m["nseg"] - 1) * m["Lo"]     # every output block in exactly one segment
    m = tool.model(4096, 4, 2, 512, 938, 112608)                        # the metric shape
    assert (m["Q"], m["Lo"], m["nseg"], m["tiles"]) == (937, 3159, 36, 9216)
    assert m["x_bytes"] == 2 * 512 * 36 * 4096 * 8 and m["y_bytes"] == 2 * 512 * 112608 * 8
    buf = (ctypes.c_int * 6)()
    lib_.tfft_geom_c(4096, 938, 112608, buf)
    assert buf[4] == 512 and buf[5] == 4 * (4096 + 4) * 8                # 512 threads, 128 KB + padding of shared memory
