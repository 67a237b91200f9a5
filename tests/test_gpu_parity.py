"""GPU parity tests (-m gpu): the CUDA path, called through the C-ABI, against
(1) golden vectors dumped from the unmodified reference, (2) the oracle port on seeded
inputs, (3) the reference's probabilities over synthetic text, with every model group resident.
Bit-exact everywhere (tolerance 0.0; north_star allows 1e-5 on probabilities)."""
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, Golden, port_replay, synthetic_streams

pytestmark = pytest.mark.gpu

TOL = 0.0   # probabilities must match bit for bit; the spec's tolerance is 1e-5
REPLAY_ALL = ("fxcm", "paq8")   # tests driven by synthetic code streams replay the big model groups instead of running them


@pytest.fixture(scope="module")
def cm():
    import cmix_b200
    cmix_b200.load_library()        # raises if the sm_100a library is missing: no fallback
    return cmix_b200


def _check_intermediates(P, g, nb):
    sx = P.debug_fetch(1, (nb, 56), np.float32)
    sel = P.debug_fetch(2, (nb, 48), np.uint32)
    lx = P.debug_fetch(3, (nb, 2), np.float32)
    assert np.array_equal(sx[:, :55], g.small_inputs[:nb, :55]), "small-model / PPMD inputs"
    cols = [i for i in range(47) if i != 12]     # selector 12 (auxiliary_context_) is produced inside the mix kernel
    assert np.array_equal(sel[:, cols], g.ctx[:nb][:, cols]), "mixer selector contexts"
    assert np.array_equal(lx[:, 0], g.small_inputs[:nb, 55]), "LSTM bit inputs"


def test_bulk_path_matches_reference_golden(cm, golden):
    g = golden
    P = cm.Predictor(g.vocab)
    p = P.code_bytes(g.stream, g.ext, g.ppmd)
    assert np.abs(p - g.p).max() <= TOL
    _check_intermediates(P, g, g.n_bytes * 8)
    lstm = P.debug_fetch(4, (256,), np.float32)
    assert np.array_equal(lstm, g.lstm[-1])
    assert P.debug_fetch(5, (1,), np.uint32)[0] == 0
    assert P.kernel_launches >= 3
    P.close()


def test_state_persists_across_calls(cm, golden_text):
    """Two bulk calls (uneven split, crossing a BPTT boundary) == one call."""
    g = golden_text
    P = cm.Predictor(g.vocab)
    k = 77
    p1 = P.code_bytes(g.stream[:k], g.ext[: k * 8], g.ppmd[:k])
    p2 = P.code_bytes(g.stream[k:], g.ext[k * 8:], g.ppmd[k:])
    assert np.array_equal(np.concatenate([p1, p2]), g.p)
    P.close()


def test_lock_step_predict_perceive_matches_reference(cm, golden_text):
    """The drop-in surface: Predict()/Perceive(bit) one bit at a time (what Encoder/Decoder call)."""
    g = golden_text
    n = 110                                  # crosses the first BPTT (byte 100)
    bits = g.bits()
    P = cm.Predictor(g.vocab)
    for t in range(n * 8):
        P.feed_external_bit(g.ext[t])
        p = P.Predict()
        assert p == g.p[t], "bit %d" % t
        if t % 8 == 7:
            P.feed_external_byte(g.ppmd[t // 8])
        P.Perceive(int(bits[t]))
    # switch to the bulk path mid-stream: same state
    rest = P.code_bytes(g.stream[n:], g.ext[n * 8:], g.ppmd[n:])
    assert np.array_equal(rest, g.p[n * 8:])
    P.close()


def test_cuda_matches_oracle_port_on_seeded_inputs(cm, port):
    """No reference needed: synthetic replay streams, ragged vocabulary, 3 BPTT rounds."""
    stream, vocab, codes, ppmd = synthetic_streams(330, seed=11)
    want, want_lstm = port_replay(port, vocab, stream, codes, ppmd, want_lstm=True)
    P = cm.Predictor(vocab, replay=REPLAY_ALL)
    got = P.code_bytes(stream, codes, ppmd)
    assert np.abs(got - want).max() <= TOL
    assert np.array_equal(P.debug_fetch(4, (256,), np.float32), want_lstm)
    P.close()


def test_edge_cases(cm, port):
    # single byte; single-symbol vocabulary (every bit hits the 0/1 override); no replay streams at all
    for stream, vocab in [
        (np.array([65], dtype=np.uint8), None),
        (np.full(40, 97, dtype=np.uint8), None),
    ]:
        if vocab is None:
            vocab = np.zeros(256, dtype=np.uint8); vocab[np.unique(stream)] = 1
        n = stream.size
        codes = np.full((n * 8, 2022), 0xFFFF, dtype=np.uint16)
        ppmd = np.tile((vocab / vocab.sum()).astype(np.float32), (n, 1))
        want = port_replay(port, vocab, stream, codes, ppmd)
        P = cm.Predictor(vocab, replay=REPLAY_ALL)
        got = P.code_bytes(stream, codes, ppmd)
        assert np.array_equal(got, want)
        P.close()
    P = cm.Predictor(np.ones(256, dtype=np.uint8))
    assert P.code_bytes(np.zeros(0, dtype=np.uint8)).size == 0     # empty input
    P.close()


def test_pretrain_then_code(cm, port):
    stream, vocab, codes, ppmd = synthetic_streams(64, seed=5)
    pre = np.frombuffer(b"the quick brown fox (jumps) over [[lazy]] dogs\n" * 3, dtype=np.uint8)
    v = np.ascontiguousarray(vocab)
    Q = port.op_create(v.ctypes.data)
    for byte in pre:
        for j in range(7, -1, -1):
            port.op_pretrain(Q, int((byte >> j) & 1))
    want = np.empty(stream.size * 8, dtype=np.float32)
    c = np.ascontiguousarray(codes); pp = np.ascontiguousarray(ppmd); s = np.ascontiguousarray(stream)
    port.op_run(Q, s.ctypes.data, s.size, c.ctypes.data, pp.ctypes.data, want.ctypes.data)
    port.op_destroy(Q)
    P = cm.Predictor(vocab, replay=REPLAY_ALL)
    P.pretrain_bytes(pre[:40].tobytes())             # bulk Pretrain ...
    for byte in pre[40:]:                            # ... and bit-by-bit Pretrain() agree
        for j in range(7, -1, -1):
            P.Pretrain(int((byte >> j) & 1))
    got = P.code_bytes(stream, codes, ppmd)
    assert np.array_equal(got, want)
    P.close()


def test_batch_of_streams_equals_individual_runs(cm):
    import torch
    runs = [synthetic_streams(48, seed=s) for s in (21, 22, 23)]
    singles = []
    for stream, vocab, codes, ppmd in runs:
        P = cm.Predictor(vocab, replay=REPLAY_ALL)
        singles.append(P.code_bytes(stream, codes, ppmd))
        P.close()
    preds = [cm.Predictor(r[1], replay=REPLAY_ALL) for r in runs]
    dev = torch.device("cuda:0")
    d_bytes = [torch.from_numpy(r[0]).to(dev) for r in runs]
    d_ext = [torch.from_numpy(r[2].view(np.int16)).to(dev) for r in runs]
    d_ppmd = [torch.from_numpy(r[3]).to(dev) for r in runs]
    d_out = [torch.empty(48 * 8, dtype=torch.float32, device=dev) for _ in runs]
    from cmix_b200.capi import code_batch_device
    code_batch_device(preds, d_bytes, 48, d_ext, d_ppmd, d_out)
    torch.cuda.synchronize()
    for o, s in zip(d_out, singles):
        assert np.array_equal(o.cpu().numpy(), s)
    for p in preds:
        p.close()


def test_host_buffer_batch_crosses_the_staging_boundary(cm, port):
    """cmixb200_code_batch: host buffers, 1024-byte double-buffered staging; 1100 bytes per stream cross it."""
    from cmix_b200.capi import code_batch
    n = 1100
    runs = [synthetic_streams(n, seed=s) for s in (31, 32)]
    want = [port_replay(port, r[1], r[0], r[2], r[3]) for r in runs]
    preds = [cm.Predictor(r[1], replay=REPLAY_ALL) for r in runs]
    outs = [np.empty(n * 8, dtype=np.float32) for _ in runs]
    code_batch(preds, [r[0] for r in runs], n, [r[2] for r in runs], [r[3] for r in runs], outs)
    for p in preds:
        p.close()
    for o, w in zip(outs, want):
        assert np.abs(o - w).max() <= TOL


def test_resident_ppmd_replaces_the_replayed_distribution(cm, golden):
    """No PPMD replay: the device model (ppmd.cuh, SURVEY a15) must reproduce the reference's
    distributions, so every Predict() still equals the reference bit for bit."""
    g = golden
    P = cm.Predictor(g.vocab)
    k = 37                                        # two bulk calls: the model's state carries over
    p = np.concatenate([P.code_bytes(g.stream[:k], g.ext[:k * 8], None), P.code_bytes(g.stream[k:], g.ext[k * 8:], None)])
    P.close()
    assert np.array_equal(p, g.p)


def test_resident_ppmd_lock_step(cm, golden_text):
    g = golden_text
    bits = g.bits()
    n = 24
    P = cm.Predictor(g.vocab)
    for t in range(n * 8):
        P.feed_external_bit(g.ext[t])
        assert P.Predict() == g.p[t], "bit %d" % t
        P.Perceive(int(bits[t]))                  # no feed_external_byte: the resident model supplies it
        if t % 8 == 7:
            assert np.array_equal(P.debug_fetch(7, (256,), np.float32), g.ppmd[t // 8])
    P.close()


@pytest.mark.parametrize("name", ["ppmd_text40k", "ppmd_bin6k", "ppmd_rand", "ppmd_rep", "ppmd_dic"])
def test_resident_ppmd_distributions_on_device(cm, name):
    """The device build of ppmd_model.h against fixtures from reference dumps (one CRC per byte)."""
    import zlib
    g = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    n = min(12000, g["stream"].size)
    import torch
    P = cm.Predictor(g["vocab"], replay=REPLAY_ALL)
    d_bytes = torch.from_numpy(g["stream"][:n].copy()).cuda()
    d_out = torch.empty(n * 8, dtype=torch.float32, device="cuda")
    P.code_bytes_device(d_bytes, n, None, None, d_out)          # one call: the debug fetch returns the last call's rows
    torch.cuda.synchronize()
    rows = P.debug_fetch(8, (n, 256), np.float32)
    P.close()
    got = np.array([zlib.crc32(rows[t].tobytes()) for t in range(n)], dtype=np.uint32)
    bad = np.nonzero(got != g["crc"][:n])[0]
    assert bad.size == 0, "first differing byte %d" % bad[0]


def test_resident_ppmd_in_a_batch(cm):
    """Several streams share one PPMD CTA (one warp each): same result as running them alone."""
    import torch
    from cmix_b200.capi import code_batch_device
    runs = [synthetic_streams(300, seed=s) for s in (41, 42, 43)]
    singles = []
    for stream, vocab, codes, _ in runs:
        P = cm.Predictor(vocab, replay=REPLAY_ALL)
        singles.append(P.code_bytes(stream, codes, None))
        P.close()
    preds = [cm.Predictor(r[1], replay=REPLAY_ALL) for r in runs]
    dev = torch.device("cuda:0")
    d_bytes = [torch.from_numpy(r[0]).to(dev) for r in runs]
    d_ext = [torch.from_numpy(r[2].view(np.int16)).to(dev) for r in runs]
    d_out = [torch.empty(300 * 8, dtype=torch.float32, device=dev) for _ in runs]
    code_batch_device(preds, d_bytes, 300, d_ext, None, d_out)
    torch.cuda.synchronize()
    for o, s in zip(d_out, singles):
        assert np.array_equal(o.cpu().numpy(), s)
    for p in preds:
        p.close()


def test_device_coder_writes_the_reference_archive_bytes(cm, port, golden_text):
    """Encoder::Encode/Flush on the device (coder.cuh): the archive body equals the host coder's over the
    reference's own probabilities, across two bulk calls, and decodes back to the input bits."""
    g = golden_text
    bits = g.bits()
    e = port.op_enc_create()
    for pr, b in zip(g.p, bits):
        port.op_enc_encode(e, float(pr), int(b))
    buf = np.zeros(g.n_bytes * 2 + 64, dtype=np.uint8)
    want = buf[:port.op_enc_finish(e, buf.ctypes.data, buf.size)].tobytes()
    port.op_enc_destroy(e)
    P = cm.Predictor(g.vocab)
    P.coder_begin(g.n_bytes * 2 + 64)
    n = 77
    P.code_bytes(g.stream[:n], g.ext[:n * 8], g.ppmd[:n])
    P.code_bytes(g.stream[n:], g.ext[n * 8:], g.ppmd[n:])
    got = P.coder_finish()
    assert got == want
    assert len(got) < g.n_bytes
    # a capacity that is too small is reported, not overrun
    P2 = cm.Predictor(g.vocab)
    P2.coder_begin(8)
    P2.code_bytes(g.stream, g.ext, g.ppmd)
    with pytest.raises(RuntimeError):
        P2.coder_finish()
    P2.close()
    # decode with the GPU predictor in lock-step (Decoder::Decode, decoder.cpp:20-39)
    coded = np.frombuffer(got, dtype=np.uint8).copy()
    d = port.op_dec_create(coded.ctypes.data, coded.size)
    D = cm.Predictor(g.vocab)
    out = np.zeros_like(bits)
    for t in range(bits.size):
        D.feed_external_bit(g.ext[t])
        b = port.op_dec_decode(d, D.Predict())
        out[t] = b
        if t % 8 == 7:
            D.feed_external_byte(g.ppmd[t // 8])
        D.Perceive(int(b))
    port.op_dec_destroy(d)
    D.close(); P.close()
    assert np.array_equal(out, bits)


def test_synthetic_text_equals_the_reference(cm):
    """2 KB of synthetic enwik-shaped text through the complete resident predictor: every Predict() equals the reference's
    (tools/make_ref_golden.py: oracle_dump over the same `cmix -n` stream), and so does the cross entropy."""
    from gen_synth import synth_text
    g = np.load(os.path.join(ROOT, "tests", "golden", "synth2k.npz"))
    assert g["stream"][5:].tobytes() == synth_text(2000, 0xE9E80002)
    P = cm.Predictor(g["vocab"])
    p = P.code_bytes(g["stream"])
    P.close()
    assert np.abs(p - g["p"]).max() <= TOL
    bits = np.unpackbits(g["stream"])
    n_bytes = g["stream"].size
    ideal = -np.log2(np.where(bits == 1, p, 1 - p).clip(1e-9, 1)).sum() / 8 / n_bytes * 8
    ideal_ref = -np.log2(np.where(bits == 1, g["p"], 1 - g["p"]).clip(1e-9, 1)).sum() / 8 / n_bytes * 8
    assert abs(ideal - ideal_ref) <= 0.001          # bits per byte within 0.001 of the reference


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "build", "cmix_b200_cli")),
                    reason="reference CLI + shim not built (make -C cmix_b200/shim)")
def test_reference_cli_round_trip(tmp_path):
    """The reference's own runner + arithmetic coder, compiled unchanged against the shim
    (INTEGRATION.md): compress then decompress through Predict()/Perceive() on the GPU."""
    from gen_synth import synth_text
    cli = os.path.join(ROOT, "build", "cmix_b200_cli")
    src = tmp_path / "in.txt"
    data = synth_text(700, 0xE9E80005)
    src.write_bytes(data)
    arc, back = tmp_path / "out.cmix", tmp_path / "back.txt"
    subprocess.run([cli, "-c", str(src), str(arc)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
    subprocess.run([cli, "-d", str(arc), str(back)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
    assert back.read_bytes() == data
    assert arc.stat().st_size < len(data)


@pytest.mark.skipif(not os.path.exists(os.path.join(ROOT, "build", "cmix_b200_cli")),
                    reason="reference CLI + shim not built (make -C cmix_b200/shim)")
def test_reference_cli_round_trip_with_dictionary(tmp_path):
    """`cmix -c <dictionary> in out`: the reference's WRT preprocessor rewrites the text and calls
    Pretrain(bit) over the dictionary (preprocessor.cpp:37-69) before the first Predict(); the shim
    buffers those bits and trains through cmixb200_pretrain_bytes."""
    import re
    from collections import Counter
    from gen_synth import synth_text
    cli = os.path.join(ROOT, "build", "cmix_b200_cli")
    data = synth_text(900, 0xE9E80006)
    words = [w for w, _ in Counter(re.findall(rb"[a-z]{3,}", data)).most_common(150)]
    dic = tmp_path / "tiny.dic"
    dic.write_bytes(b"\n".join(words) + b"\n")
    src = tmp_path / "in.txt"
    src.write_bytes(data)
    arc, back = tmp_path / "out.cmix", tmp_path / "back.txt"
    subprocess.run([cli, "-c", str(dic), str(src), str(arc)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
    subprocess.run([cli, "-d", str(dic), str(arc), str(back)], check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL, timeout=600)
    assert back.read_bytes() == data
    assert arc.stat().st_size < len(data)
