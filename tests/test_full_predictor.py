"""The complete predictor with every model group resident (SURVEY §8 rows a1-a18): no replayed inputs anywhere.

Fixtures (tools/make_full_golden.py) come from dumps of the unmodified reference: Predictor::Predict() of every bit plus a
CRC32 per 4096 bits over its FXCM codes and over its PAQ8 codes.
CPU (-m "not gpu"): the host build of the PAQ8 model (tools/paq8_check.cpp) against the PAQ8 CRCs.
GPU (-m gpu): bytes in, probabilities out through the C-ABI; must equal the reference's probabilities bit for bit
(tolerance 0; north_star allows 1e-5), bulk and lock-step, and the generated FXCM / PAQ8 codes must match the CRCs."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from conftest import ROOT


def _load(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def paq8_check(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("p8") / "paq8_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-ffp-contract=off", "-I", os.path.join(ROOT, "cmix_b200", "csrc"),
                    os.path.join(ROOT, "tools", "paq8_check.cpp"), "-o", exe], check=True)
    return exe


@pytest.mark.parametrize("name", ["full_text", "full_bin"])
def test_paq8_host_build_matches_reference_codes(paq8_check, tmp_path, name):
    g = _load(name)
    n = 2048                                           # 4 CRC blocks: ~5 s of CPU per fixture
    prefix = str(tmp_path / "d")
    g["stream"][:n].tofile(prefix + ".stream")
    crc_out = prefix + ".crc"
    r = subprocess.run([paq8_check, prefix, "-", str(n), crc_out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(crc_out, dtype=np.uint32)
    assert np.array_equal(got, g["crc_p8"][:got.size]) and got.size == n * 8 // 4096


def test_paq8_tables_are_the_reference_tables():
    """The hex tables in paq8_host.h against what the reference's own initialisers produce (tools/make_ref_golden.py)."""
    from make_paq8_tables import differences
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_tables.npz"))
    want = {k[len("paq8_"):]: z[k].tobytes().hex() for k in z.files if k.startswith("paq8_")}
    assert len(want) == 15
    assert differences(want) == []


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def cm():
    import cmix_b200
    cmix_b200.load_library()
    return cmix_b200


def _run_resident(cm, g, dictionary=None, pretrain=None, piece=2048, n=None):
    stream = g["stream"] if n is None else g["stream"][:n]
    P = cm.Predictor(g["vocab"], dictionary_path=dictionary)
    if pretrain is not None:
        P.pretrain_bytes(pretrain)
    ps, crc_fx, crc_p8, first = [], [], [], None
    for off in range(0, stream.size, piece):
        part = stream[off:off + piece]
        ps.append(P.code_bytes(part, None, None))
        ext = P.debug_fetch(10, (part.size * 8, 2022), np.uint16)
        if first is None:
            first = ext[:64].copy()
        for b in range(0, ext.shape[0], 4096):
            crc_fx.append(zlib.crc32(np.ascontiguousarray(ext[b:b + 4096, :431]).tobytes()))
            crc_p8.append(zlib.crc32(np.ascontiguousarray(ext[b:b + 4096, 431:]).tobytes()))
    P.close()
    return np.concatenate(ps), np.array(crc_fx, dtype=np.uint32), np.array(crc_p8, dtype=np.uint32), first


def _assert_matches(g, p, crc_fx, crc_p8, first):
    bad = np.argwhere(first != g["first_codes"])
    assert bad.size == 0, "codes of the first 64 bits: first differing (bit, slot) %s" % (bad[:1],)
    k = crc_fx.size
    b = np.nonzero(crc_fx != g["crc_fx"][:k])[0]
    assert b.size == 0, "FXCM codes: first differing 4096-bit block %d" % b[0]
    b = np.nonzero(crc_p8 != g["crc_p8"][:k])[0]
    assert b.size == 0, "PAQ8 codes: first differing 4096-bit block %d" % b[0]
    d = np.nonzero(p != g["p"][:p.size])[0]
    assert d.size == 0, "Predict(): first differing bit %d (%.9g vs %.9g)" % (d[0], p[d[0]], g["p"][d[0]])


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["full_text", "full_bin"])
def test_everything_resident_equals_the_reference(cm, name):
    g = _load(name)
    p, crc_fx, crc_p8, first = _run_resident(cm, g)
    _assert_matches(g, p, crc_fx, crc_p8, first)
    bits = np.unpackbits(g["stream"])
    bpc = -np.log2(np.where(bits == 1, p, 1 - p).clip(1e-9, 1)).sum() / g["stream"].size
    bpc_ref = -np.log2(np.where(bits == 1, g["p"], 1 - g["p"]).clip(1e-9, 1)).sum() / g["stream"].size
    assert abs(bpc - bpc_ref) <= 0.001                 # north_star: compressed bits per byte within 0.001 of the reference


@pytest.mark.gpu
def test_everything_resident_with_dictionary_and_pretraining(cm, english_dic):
    """cmix -c english.dic in out: WRT code words in the stream, Pretrain() over header + dictionary before the first bit."""
    g = _load("full_wrt")
    d = open(english_dic, "rb").read()
    pre = bytes([0, (len(d) >> 24) & 255, (len(d) >> 16) & 255, (len(d) >> 8) & 255, len(d) & 255]) + d.replace(b"\n", b" ")
    p, crc_fx, crc_p8, first = _run_resident(cm, g, dictionary=english_dic, pretrain=pre, n=2048)
    _assert_matches(g, p, crc_fx, crc_p8, first)


@pytest.mark.gpu
def test_everything_resident_lock_step(cm):
    """Predict()/Perceive(bit) one bit at a time (the decoder's order), then the bulk kernels mid-stream."""
    g = _load("full_text")
    bits = np.unpackbits(g["stream"])
    P = cm.Predictor(g["vocab"])
    n = 24
    for t in range(n * 8):
        assert P.Predict() == g["p"][t], "bit %d" % t
        P.Perceive(int(bits[t]))
    rest = P.code_bytes(g["stream"][n:512], None, None)
    P.close()
    assert np.array_equal(rest, g["p"][n * 8:512 * 8])


@pytest.mark.gpu
def test_unmodelled_block_fails_loudly(cm):
    """PAQ8's image / audio / JPEG sub-models are not resident: a stream in which its block parser would validate such a header
    must make the call fail (CMIXB200_ERR_UNSUPPORTED), never return different predictions silently."""
    g = _load("full_text")
    text = g["stream"][:700].copy()
    jpeg = np.frombuffer(bytes([0xFF, 0xD8, 0xFF, 0xE0, 0x00, 0x10]) + b"JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00", dtype=np.uint8)
    stream = np.concatenate([text[:300], jpeg, text[300:]])
    P = cm.Predictor(np.ones(256, dtype=np.uint8))
    with pytest.raises(RuntimeError, match="image / audio / JPEG"):
        P.code_bytes(stream, None, None)
    P.close()
