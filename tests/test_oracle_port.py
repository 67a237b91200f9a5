"""CPU tests (-m "not gpu"): pin the oracle restatement against the reference's own outputs."""
import ctypes
import os
import re
import subprocess

import numpy as np
import pytest

from conftest import ROOT, port_replay, synthetic_streams


def test_port_matches_reference_bit_for_bit(port, golden):
    g = golden
    vocab = np.ascontiguousarray(g.vocab)
    P = port.op_create(vocab.ctypes.data)
    bits = g.bits()
    inp = np.zeros(2078, np.float32); mix = np.zeros(47, np.float32); ctx = np.zeros(47, np.uint32); lp = np.zeros(256, np.float32)
    cols = list(range(3)) + list(range(2025, 2078))
    for t in range(bits.size):
        e = np.ascontiguousarray(g.ext[t])
        p = port.op_predict(P, e.ctypes.data)
        port.op_get_inputs(P, inp.ctypes.data)
        port.op_get_mixer_outputs(P, mix.ctypes.data)
        port.op_get_mixer_contexts(P, ctx.ctypes.data)
        assert np.float32(p) == g.p[t], "Predict() differs at bit %d" % t
        assert np.array_equal(inp[cols], g.small_inputs[t]), "small-model inputs differ at bit %d" % t
        if t < 64:
            assert np.array_equal(inp, g.inputs_first64[t])
        assert np.array_equal(mix, g.mix[t]), "mixer outputs differ at bit %d" % t
        assert np.array_equal(ctx, g.ctx[t]), "mixer selectors differ at bit %d" % t
        pp = np.ascontiguousarray(g.ppmd[t // 8])
        port.op_perceive(P, int(bits[t]), pp.ctypes.data)
        if t % 8 == 7:
            port.op_get_lstm_probs(P, lp.ctypes.data)
            assert np.array_equal(lp, g.lstm[t // 8]), "LSTM byte distribution differs after byte %d" % (t // 8)
    port.op_destroy(P)


def _encode(port, p, bits):
    e = port.op_enc_create()
    for pr, b in zip(p, bits):
        port.op_enc_encode(e, float(pr), int(b))
    buf = np.zeros(len(bits) // 4 + 64, dtype=np.uint8)
    n = port.op_enc_finish(e, buf.ctypes.data, buf.size)
    port.op_enc_destroy(e)
    return buf[:n].copy()


def test_coder_round_trip_through_the_port(port, golden_text):
    """encode -> decode with the predictor replayed in lock-step gives the bits back."""
    g = golden_text
    bits = g.bits()
    coded = _encode(port, g.p, bits)
    assert coded.size < g.n_bytes            # it actually compresses
    vocab = np.ascontiguousarray(g.vocab)
    P = port.op_create(vocab.ctypes.data)
    d = port.op_dec_create(coded.ctypes.data, coded.size)
    got = np.zeros_like(bits)
    for t in range(bits.size):
        e = np.ascontiguousarray(g.ext[t])
        p = port.op_predict(P, e.ctypes.data)
        b = port.op_dec_decode(d, p)
        got[t] = b
        pp = np.ascontiguousarray(g.ppmd[t // 8])
        port.op_perceive(P, b, pp.ctypes.data)
    port.op_dec_destroy(d)
    port.op_destroy(P)
    assert np.array_equal(got, bits)


def test_archive_matches_reference_cli(port, golden_text):
    """header + coder(p-stream) == the archive the unmodified reference CLI writes (cmix -n) for the file whose stream
    (5-byte DEFAULT block header + file) is text208's; tools/make_ref_golden.py stored that archive."""
    g = golden_text
    ref = np.fromfile(os.path.join(ROOT, "tests", "golden", "text208.cmix"), dtype=np.uint8)
    n = g.n_bytes
    header = np.array([(n >> (8 * i)) & 0xFF for i in (4, 3, 2, 1, 0)], dtype=np.uint8)   # runner.cpp:34-44, < 10000 B: no vocab
    mine = np.concatenate([header, _encode(port, g.p, g.bits())])
    assert np.array_equal(mine, ref)


def test_port_is_deterministic_and_learns(port):
    stream, vocab, codes, ppmd = synthetic_streams(96, seed=7)
    p1 = port_replay(port, vocab, stream, codes, ppmd)
    p2 = port_replay(port, vocab, stream, codes, ppmd)
    assert np.array_equal(p1, p2)
    bits = np.unpackbits(stream)
    pr = np.where(bits == 1, p1, 1 - p1).clip(1e-6, 1)
    assert -np.log2(pr).mean() < 0.9             # better than 1 bit/bit: the mixer uses its inputs


def test_exact_math_matches_libm(port, tmp_path):
    """cmix_b200/csrc/exact_math.h (host build) == glibc expf/tanhf on a dense sample.
    (tools/exact_math_sweep.cpp checks all 2^32 inputs; 0 mismatches recorded in DESIGN.md.)"""
    src = tmp_path / "xm.cpp"
    src.write_text('#include "%s/cmix_b200/csrc/exact_math.h"\n'
                   'extern "C" float t_expf(float x){return xm_expf(x);} extern "C" float t_tanhf(float x){return xm_tanhf(x);}\n'
                   'extern "C" float t_logistic(float x){return xm_logistic(x);}\n'
                   'extern "C" void t_many(const float* x, float* e, float* t, float* l, int n){for(int i=0;i<n;++i){e[i]=xm_expf(x[i]);t[i]=xm_tanhf(x[i]);l[i]=xm_logistic(x[i]);}}\n' % ROOT)
    so = tmp_path / "libxm.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-fPIC", "-shared", str(src), "-o", str(so), "-lm"], check=True)
    lib = ctypes.CDLL(str(so))
    lib.t_many.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_int]
    rng = np.random.default_rng(1)
    xs = np.concatenate([
        rng.uniform(-110, 90, 400000), rng.uniform(-25, 25, 400000), rng.normal(0, 1, 200000),
        np.frombuffer(rng.integers(0, 2**32, 200000, dtype=np.uint32).tobytes(), dtype=np.float32).astype(np.float64),
    ]).astype(np.float32)
    xs = xs[np.isfinite(xs)]
    e = np.empty_like(xs); t = np.empty_like(xs); l = np.empty_like(xs)
    lib.t_many(xs.ctypes.data, e.ctypes.data, t.ctypes.data, l.ctypes.data, xs.size)
    port.op_libm_expf.restype = ctypes.c_float
    for i in rng.integers(0, xs.size, 20000):
        x = float(xs[i])
        assert np.float32(port.op_libm_expf(x)).tobytes() == e[i].tobytes(), x
        assert np.float32(port.op_libm_tanhf(x)).tobytes() == t[i].tobytes(), x
        assert np.float32(port.op_logistic(x)).tobytes() == l[i].tobytes(), x


def test_c_abi_library_exports_every_declared_symbol():
    """The drop-in boundary loads on a CPU-only box and exports all of include/cmixb200.h."""
    import cmix_b200
    if not os.path.exists(cmix_b200.LIB_PATH):
        cmix_b200.build_library()
    lib = ctypes.CDLL(cmix_b200.LIB_PATH)
    header = open(os.path.join(ROOT, "include", "cmixb200.h")).read()
    names = sorted(set(re.findall(r"\b(cmixb200_[a-z_0-9]+)\s*\(", header)))
    assert len(names) >= 14
    for n in names:
        assert hasattr(lib, n), n


def test_no_cpu_fallback_without_a_gpu():
    """On a box without a GPU the product must fail loudly, not fall back."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import cmix_b200
    if not os.path.exists(cmix_b200.LIB_PATH):
        cmix_b200.build_library()
    with pytest.raises(RuntimeError):
        cmix_b200.Predictor(np.ones(256, dtype=np.uint8))


def test_product_does_not_touch_the_oracle():
    """Nothing under cmix_b200/ or include/ may include, import, link, open or execute anything under oracle/:
    the oracle is test infrastructure (only tests/, smoke() and bench.py's CPU-baseline legs may use it)."""
    import re
    forbidden = re.compile(r"oracle/|oracle\\|liboracle|oracle_port|oracle_dump|import\s+oracle|from\s+oracle|oracle_io|load_port")
    for base in ("cmix_b200", "include"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, base)):
            for f in files:
                if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")) or f == "Makefile":
                    text = open(os.path.join(dirpath, f), errors="ignore").read()
                    m = forbidden.search(text)
                    assert m is None, "%s mentions %r" % (os.path.join(dirpath, f), m.group(0))
