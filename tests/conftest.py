import lzma
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run on the GPU box with -m gpu)")


class Golden:
    """A fixture written by tools/make_golden.py from the unmodified reference."""

    def __init__(self, name):
        z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
        self.stream = z["stream"]
        self.vocab = z["vocab"]
        self.p = z["p"]
        self.ext = z["ext"]
        self.ppmd = z["ppmd"]
        self.lstm = z["lstm"]
        self.mix = z["mix"]
        self.ctx = z["ctx"]
        self.small_inputs = z["small_inputs"]      # layer-0 inputs 0..2 and 2025..2077
        self.inputs_first64 = z["inputs_first64"]
        self.n_bytes = int(self.stream.size)

    def bits(self):
        return np.unpackbits(self.stream)


@pytest.fixture(scope="session", params=["text208", "binary120"])
def golden(request):
    return Golden(request.param)


@pytest.fixture(scope="session")
def golden_text():
    return Golden("text208")


@pytest.fixture(scope="session")
def english_dic(tmp_path_factory):
    """The reference's WRT dictionary (`cmix -c english.dic`), stored xz-compressed by tools/make_ref_golden.py."""
    path = tmp_path_factory.mktemp("dic") / "english.dic"
    with lzma.open(os.path.join(ROOT, "tests", "golden", "english.dic.xz")) as f:
        path.write_bytes(f.read())
    return str(path)


@pytest.fixture(scope="session")
def port():
    """The CPU restatement (oracle/port), built on demand with g++."""
    so = os.path.join(ROOT, "oracle", "_ref", "liboracle_port.so")
    if not os.path.exists(so):
        subprocess.run(["make", "-C", os.path.join(ROOT, "oracle"), "port"], check=True)
    from oracle_io import load_port
    return load_port()


def port_replay(lib, vocab, stream, ext, ppmd, want_lstm=False):
    """Run the port over a byte stream with replayed model streams; returns p per bit."""
    vocab = np.ascontiguousarray(vocab, dtype=np.uint8)
    stream = np.ascontiguousarray(stream, dtype=np.uint8)
    ext = np.ascontiguousarray(ext, dtype=np.uint16)
    ppmd = np.ascontiguousarray(ppmd, dtype=np.float32)
    P = lib.op_create(vocab.ctypes.data)
    out = np.empty(stream.size * 8, dtype=np.float32)
    lib.op_run(P, stream.ctypes.data, stream.size, ext.ctypes.data, ppmd.ctypes.data, out.ctypes.data)
    lstm = None
    if want_lstm:
        lstm = np.empty(256, dtype=np.float32)
        lib.op_get_lstm_probs(P, lstm.ctypes.data)
    lib.op_destroy(P)
    return (out, lstm) if want_lstm else out


def synthetic_streams(n_bytes, seed, vocab_lo=32, vocab_hi=127):
    """Seeded stand-ins for the replayed PAQ8/FXCM/PPMD streams (no reference needed)."""
    rng = np.random.default_rng(seed)
    stream = rng.integers(vocab_lo, vocab_hi, size=n_bytes, dtype=np.uint8)
    stream[rng.random(n_bytes) < 0.15] = 32
    vocab = np.zeros(256, dtype=np.uint8)
    vocab[np.unique(stream)] = 1
    bits = np.unpackbits(stream)
    # codes correlated with the coded bit so that the mixer has something to learn
    noise = rng.normal(0.0, 1.2, size=(bits.size, 2022)).astype(np.float32)
    skill = rng.uniform(0.0, 1.5, size=2022).astype(np.float32)
    logit = noise + skill * (2.0 * bits[:, None].astype(np.float32) - 1.0)
    codes = np.clip(np.rint(4095.0 / (1.0 + np.exp(-logit))), 0, 4095).astype(np.uint16)
    codes[:, 429:431] = 0xFFFF            # slots the reference never writes stay at 0.5 (SURVEY App. B #19)
    ppmd = rng.gamma(0.3, 1.0, size=(n_bytes, 256)).astype(np.float32) + 1e-6
    nxt = np.roll(stream, -1)
    ppmd[np.arange(n_bytes), nxt] += rng.uniform(0, 8, size=n_bytes).astype(np.float32)
    ppmd *= vocab[None, :]
    ppmd = (ppmd / ppmd.sum(axis=1, keepdims=True)).astype(np.float32)
    return stream, vocab, codes, ppmd
