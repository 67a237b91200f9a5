"""Fixtures that let the suite compare with the unmodified reference without its sources or binaries at test time.

    make -C oracle ref REF=<cmix checkout>
    python tools/make_ref_golden.py <cmix checkout>

writes under tests/golden/:
    english.dic.xz   the reference's WRT dictionary (dictionary/english.dic), xz-compressed: input data of `cmix -c`
    ref_tables.npz   the constant tables its initialisers produce: PAQ8's (tools/make_paq8_tables.py) and FXCM's wrt_2b/3b/4b
    text208.cmix     the archive the reference CLI (oracle/_ref/cmix_strict -n) writes for text208's file
    synth2k.npz      stream, vocabulary and Predict() of every bit of oracle/_ref/oracle_dump over gen_synth text
                     (2000 bytes, seed 0xE9E80002, no preprocessing)
"""
import lzma
import os
import re
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
GOLDEN = os.path.join(ROOT, "tests", "golden")
REF_BIN = os.path.join(ROOT, "oracle", "_ref")


def fxcm_tables(src):
    text = open(os.path.join(src, "src", "models", "fxcmv1.cpp")).read()
    out = {}
    for name in ("wrt_2b", "wrt_3b", "wrt_4b"):
        body = re.sub(r"//.*", "", re.search(name + r"\[\d+\]\s*=\s*\{(.*?)\};", text, re.S).group(1))
        out["fxcm_" + name] = np.array([int(x) for x in re.findall(r"\d+", body)], dtype=np.uint8)
    return out


def main():
    src = sys.argv[1]
    import make_paq8_tables
    from gen_synth import synth_text
    from oracle_io import Dump

    dic = open(os.path.join(src, "dictionary", "english.dic"), "rb").read()
    with lzma.open(os.path.join(GOLDEN, "english.dic.xz"), "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(dic)

    make_paq8_tables.REF = os.path.join(src, "src", "models", "paq8.cpp")
    tables = {"paq8_" + k: np.frombuffer(bytes.fromhex(v), dtype=np.uint8) for k, v in make_paq8_tables.tables().items()}
    tables.update(fxcm_tables(src))
    np.savez_compressed(os.path.join(GOLDEN, "ref_tables.npz"), **tables)

    with tempfile.TemporaryDirectory() as tmp:
        g = np.load(os.path.join(GOLDEN, "text208.npz"))
        open(os.path.join(tmp, "in.bin"), "wb").write(g["stream"][5:].tobytes())     # the stream carries the 5-byte block header
        subprocess.run([os.path.join(REF_BIN, "cmix_strict"), "-n", os.path.join(tmp, "in.bin"), os.path.join(GOLDEN, "text208.cmix")],
                       check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)

        open(os.path.join(tmp, "in.txt"), "wb").write(synth_text(2000, 0xE9E80002))
        subprocess.run([os.path.join(REF_BIN, "oracle_dump"), "dump", "n", os.path.join(tmp, "in.txt"), os.path.join(tmp, "d"), "0"],
                       check=True, stdout=subprocess.DEVNULL, stderr=subprocess.DEVNULL)
        d = Dump(os.path.join(tmp, "d"))
        np.savez_compressed(os.path.join(GOLDEN, "synth2k.npz"), stream=d.stream, vocab=d.vocab, p=d.p)
    for f in ("english.dic.xz", "ref_tables.npz", "text208.cmix", "synth2k.npz"):
        print(f, os.path.getsize(os.path.join(GOLDEN, f)), "bytes")


if __name__ == "__main__":
    main()
