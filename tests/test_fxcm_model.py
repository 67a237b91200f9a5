"""The resident FXCM model (SURVEY §8 row a14, cmix_b200/csrc/fxcm_model.h).

CPU (-m "not gpu"): the host build of the model is run by tools/fxcm_check.cpp over fixtures made from dumps of the
unmodified reference (tools/make_fxcm_golden.py): every one of the 431 exported 12-bit codes of every bit must match
(one CRC32 per 4096 bits). GPU (-m gpu): the same fixtures through the device kernels with PPMD, LSTM and FXCM all
resident, so the LSTM feedback FXCM consumes is the device's own."""
import os
import subprocess
import zlib

import numpy as np
import pytest

from conftest import ROOT, Golden

FIXTURES = ["fxcm_text", "fxcm_bin", "fxcm_wrt"]


def _load(name):
    z = np.load(os.path.join(ROOT, "tests", "golden", name + ".npz"))
    return {k: z[k] for k in z.files}


@pytest.fixture(scope="module")
def fxcm_check(tmp_path_factory):
    exe = str(tmp_path_factory.mktemp("fx") / "fxcm_check")
    subprocess.run(["g++", "-O2", "-std=c++17", "-I", os.path.join(ROOT, "cmix_b200", "csrc"),
                    os.path.join(ROOT, "tools", "fxcm_check.cpp"), "-o", exe], check=True)
    return exe


@pytest.mark.parametrize("name", FIXTURES)
def test_host_build_matches_reference_codes(fxcm_check, english_dic, tmp_path, name):
    g = _load(name)
    use_dict = bool(g["dictionary"][0])
    prefix = str(tmp_path / "d")
    g["stream"].tofile(prefix + ".stream")
    g["lstmfx"].tofile(prefix + ".lstmfx.u32")
    crc_out = prefix + ".crc"
    r = subprocess.run([fxcm_check, prefix, english_dic if use_dict else "-", str(g["stream"].size), crc_out], capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    got = np.fromfile(crc_out, dtype=np.uint32)
    bad = np.nonzero(got != g["crc"])[0]
    assert got.size == g["crc"].size and bad.size == 0, "first differing 4096-bit block: %s" % (bad[:1],)


def test_tables_are_the_reference_tables():
    """The byte-class tables are spelled as digit strings in fxcm_host.h; compare them with the reference's (tools/make_ref_golden.py)."""
    import re
    ref = np.load(os.path.join(ROOT, "tests", "golden", "ref_tables.npz"))
    mine = open(os.path.join(ROOT, "cmix_b200", "csrc", "fxcm_host.h")).read()
    for theirs, ours in (("wrt_2b", "wrt2"), ("wrt_3b", "wrt3"), ("wrt_4b", "wrt4")):
        want = ref["fxcm_" + theirs].tolist()
        assert len(want) == 256
        m = re.search(r"fill_digits\(T\." + ours + r", 256,(.*?)\);", mine, re.S)
        got = [int(c, 16) for c in "".join(re.findall(r'"(.*?)"', m.group(1))).replace(" ", "")]
        assert got == want, theirs


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def cm():
    import cmix_b200
    cmix_b200.load_library()
    return cmix_b200


def _device_code_crcs(cm, g, dictionary=None, pretrain=None, piece=2048):
    P = cm.Predictor(g["vocab"], dictionary_path=dictionary)
    if pretrain is not None:
        P.pretrain_bytes(pretrain)
    stream = g["stream"]
    crcs, crc, done = [], 0, 0
    first = None
    for off in range(0, stream.size, piece):
        part = stream[off:off + piece]
        P.code_bytes(part, None, None)                         # PAQ8 slots stay at 0.5: FXCM does not depend on the mixer
        ext = P.debug_fetch(10, (part.size * 8, 2022), np.uint16)
        if first is None:
            first = ext[:64, :431].copy()
        codes = np.ascontiguousarray(ext[:, :431])
        for b in range(0, codes.shape[0], 4096):
            crcs.append(zlib.crc32(codes[b:b + 4096].tobytes()))
    P.close()
    return np.array(crcs, dtype=np.uint32), first


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["fxcm_text", "fxcm_bin"])
def test_device_fxcm_chain_matches_reference_codes(cm, name):
    g = _load(name)
    got, first = _device_code_crcs(cm, g)
    assert np.array_equal(first, g["first_codes"]), "codes of the first 64 bits"
    bad = np.nonzero(got != g["crc"])[0]
    assert bad.size == 0, "first differing 4096-bit block %d" % bad[0]


@pytest.mark.gpu
def test_device_fxcm_with_dictionary_and_pretraining(cm, english_dic):
    """cmix -c english.dic: WRT code words in the stream, Pretrain() over header + dictionary before the first bit."""
    g = _load("fxcm_wrt")
    d = open(english_dic, "rb").read()
    pre = bytes([0, (len(d) >> 24) & 255, (len(d) >> 16) & 255, (len(d) >> 8) & 255, len(d) & 255]) + d.replace(b"\n", b" ")
    n = 2048                                                   # 3 CRC blocks... keep the GPU test short: pretraining dominates
    g = dict(g); g["stream"] = g["stream"][:n]
    got, first = _device_code_crcs(cm, g, dictionary=english_dic, pretrain=pre)
    assert np.array_equal(first, g["first_codes"])
    assert np.array_equal(got, g["crc"][:got.size])


@pytest.mark.gpu
def test_resident_fxcm_in_the_full_predictor(cm):
    """Golden vectors of the whole predictor: with FXCM resident (PAQ8 replayed) Predict() still equals the reference, and the
    generated codes equal the reference's FXCM outputs slot by slot."""
    for name in ("text208", "binary120"):
        g = Golden(name)
        P = cm.Predictor(g.vocab)
        p = P.code_bytes(g.stream, g.ext, None)
        ext = P.debug_fetch(10, (g.n_bytes * 8, 2022), np.uint16)
        P.close()
        bad = np.argwhere(ext[:, :431] != g.ext[:, :431])
        assert bad.size == 0, "first differing (bit, slot): %s" % (bad[:1],)
        assert np.array_equal(ext[:, 431:], g.ext[:, 431:]), "replayed PAQ8 slots are passed through"
        assert np.array_equal(p, g.p)


@pytest.mark.gpu
def test_resident_fxcm_lock_step(cm):
    g = Golden("text208")
    bits = g.bits()
    P = cm.Predictor(g.vocab)
    for t in range(40 * 8):
        P.feed_external_bit(g.ext[t])
        codes = P.debug_fetch(11, (2022,), np.uint16)
        assert np.array_equal(codes[:431], g.ext[t, :431]), "bit %d" % t
        assert P.Predict() == g.p[t], "bit %d" % t
        P.Perceive(int(bits[t]))
    rest = P.code_bytes(g.stream[40:], g.ext[40 * 8:], None)   # switch to the bulk kernels mid-stream
    P.close()
    assert np.array_equal(rest, g.p[40 * 8:])
