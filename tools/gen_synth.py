"""Seeded synthetic corpora shaped like the BASELINE.json configs (SURVEY.md §8d).

    python tools/gen_synth.py text 100000 out.txt [seed]
    python tools/gen_synth.py binary 100000 out.bin [seed]

text: enwik8/enwik9 shape. Words are drawn Zipf(s=1.07) over the ranks of the WRT dictionary
(english.dic, rank = line number; stored as tests/golden/english.dic.xz) so that `cmix -c english.dic`
finds dictionary hits. Sentences of
3+Poisson(14) words, 12 % capitalised starts, punctuation, [[wiki links]], entities, numbers,
paragraphs, plus the wiki structures the text models key on (headings, lists, tables, templates,
<math>/<nowiki>/<pre>, external links, bold/italic), every ~4 KB wrapped in a <page> element.
Bytes are ASCII 0x0A, 0x20-0x7E only.

binary: alternating 64 KiB blocks of (i) x86-64 ELF-like code with repeating E8/E9/0F 8x rel32
targets and (ii) baseline-JPEG files whose scan is a real Huffman-coded stream (standard tables,
random DCT coefficients, FF00 stuffing) so that a JPEG parser sees MCUs.
"""
import lzma
import os
import sys
import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DICT_PATH = os.path.join(ROOT, "tests", "golden", "english.dic.xz")


def _words():
    with lzma.open(DICT_PATH) as f:
        return [w for w in f.read().decode("latin-1").split("\n") if w and w.isascii() and w.isalpha()]


class _TextGen:
    def __init__(self, seed):
        self.rng = np.random.default_rng(seed)
        self.words = _words()
        ranks = np.arange(1, len(self.words) + 1, dtype=np.float64)
        pz = ranks ** -1.07
        self.cdf = np.cumsum(pz / pz.sum())

    def draw(self, n):
        return [self.words[min(i, len(self.words) - 1)] for i in np.searchsorted(self.cdf, self.rng.random(n))]

    def word(self):
        return self.draw(1)[0]

    def sentence(self):
        rng = self.rng
        n_w = 3 + int(rng.poisson(14))
        toks = []
        for k, w in enumerate(self.draw(n_w)):
            r = rng.random()
            if r < 0.03:
                w = "[[" + w + (("|" + self.word()) if rng.random() < 0.3 else "") + "]]" + ("s" if rng.random() < 0.1 else "")
            elif r < 0.05:
                y = int(rng.integers(1, 2100))
                w = str(y) if rng.random() < 0.6 else ("%d,%03d" % (y, int(rng.integers(0, 1000))) if rng.random() < 0.5 else "%d.%d" % (y % 100, int(rng.integers(0, 100))))
            elif r < 0.053:
                w = ("&quot;" + w + "&quot;") if rng.random() < 0.7 else (w + " &amp; " + self.word())
            elif r < 0.06:
                q = "'''" if rng.random() < 0.4 else "''"
                w = q + w + q
            elif r < 0.063:
                w = "[http://www." + self.word() + ".org/" + self.word() + " " + self.word() + "]"
            elif r < 0.066:
                w = "&lt;math&gt;" + self.word()[:1] + "^2 + " + str(int(rng.integers(1, 99))) + "&lt;/math&gt;"
            elif r < 0.068:
                w = "{{" + self.word() + "|" + self.word() + "=" + self.word() + "}}"
            elif r < 0.07:
                w = self.word() + "'s"
            elif r < 0.072:
                w = self.word() + "-" + self.word()
            elif r < 0.074:
                w = w.upper()
            if k == 0 or rng.random() < 0.04:
                w = w[:1].upper() + w[1:]
            if k < n_w - 1 and rng.random() < 0.08:
                w += str(rng.choice([",", ",", ";", ":", " (", ")", " \"", "\""]))
            toks.append(w)
        return " ".join(toks) + str(rng.choice([".", ".", ".", ".", "?", "!"]))

    def paragraph(self):
        n_words = 60 + int(self.rng.geometric(1.0 / 120))
        out, n = [], 0
        while n < n_words:
            s = self.sentence()
            out.append(s)
            n += s.count(" ") + 1
        return " ".join(out) + "\n\n"

    def block(self):
        rng = self.rng
        r = rng.random()
        if r < 0.62:
            return self.paragraph()
        if r < 0.70:
            lvl = "=" * int(rng.integers(2, 4))
            return lvl + " " + " ".join(w.capitalize() for w in self.draw(1 + int(rng.integers(3)))) + " " + lvl + "\n"
        if r < 0.80:
            return "".join(("*" * int(rng.integers(1, 3))) + " " + ("[[" + self.word() + "]] - " if rng.random() < 0.4 else "") +
                           " ".join(self.draw(2 + int(rng.integers(8)))) + "\n" for _ in range(2 + int(rng.integers(6)))) + "\n"
        if r < 0.87:
            cols = 2 + int(rng.integers(3))
            rows = ["{| class=\"wikitable\"\n"]
            for _ in range(2 + int(rng.integers(5))):
                rows.append("|-\n| " + " || ".join(self.word() if rng.random() < 0.6 else str(int(rng.integers(0, 5000))) for _ in range(cols)) + "\n")
            rows.append("|}\n\n")
            return "".join(rows)
        if r < 0.91:
            return "{{" + self.word().capitalize() + "\n" + "".join("| " + self.word() + " = " + " ".join(self.draw(1 + int(rng.integers(3)))) + "\n" for _ in range(2 + int(rng.integers(4)))) + "}}\n"
        if r < 0.94:
            return "&lt;pre&gt;\n" + "".join("  " + " ".join(self.draw(3 + int(rng.integers(5)))) + "\n" for _ in range(2 + int(rng.integers(3)))) + "&lt;/pre&gt;\n\n"
        if r < 0.96:
            return "&lt;nowiki&gt;" + " ".join(self.draw(4)) + "&lt;/nowiki&gt;\n\n"
        if r < 0.98:
            return "[[Category:" + " ".join(w.capitalize() for w in self.draw(2)) + "]]\n[[Image:" + self.word() + ".jpg|thumb|" + " ".join(self.draw(5)) + "]]\n"
        return ":" + " ".join(self.draw(6)) + "\n#REDIRECT [[" + self.word().capitalize() + "]]\n"

    def page(self, ident):
        rng = self.rng
        title = " ".join(w.capitalize() for w in self.draw(1 + int(rng.integers(3))))
        head = ("  <page>\n    <title>%s</title>\n    <id>%d</id>\n    <revision>\n      <id>%d</id>\n      <timestamp>20%02d-%02d-%02dT%02d:%02d:%02dZ</timestamp>\n"
                "      <contributor>\n        <username>%s</username>\n        <id>%d</id>\n      </contributor>\n      <text xml:space=\"preserve\">"
                % (title, ident, 15900000 + ident * 7, rng.integers(2, 7), rng.integers(1, 13), rng.integers(1, 29), rng.integers(0, 24),
                   rng.integers(0, 60), rng.integers(0, 60), self.word().capitalize(), rng.integers(1, 99999)))
        body, n = [], 0
        while n < 3500:
            b = self.block()
            body.append(b)
            n += len(b)
        return head + "".join(body) + "</text>\n    </revision>\n  </page>\n"


def synth_text(n_bytes, seed=0xE9E80001):
    g = _TextGen(seed)
    out, size, ident = [], 0, 0
    while size < n_bytes:
        ident += 1
        s = g.page(ident)
        out.append(s)
        size += len(s)
    return "".join(out).encode("ascii")[:n_bytes]


# ---- baseline JPEG with a real Huffman-coded scan (ITU T.81 Annex K tables) ----
_DC_L_BITS = [0, 1, 5, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0, 0, 0]
_DC_C_BITS = [0, 3, 1, 1, 1, 1, 1, 1, 1, 1, 1, 0, 0, 0, 0, 0]
_DC_VALS = list(range(12))
_AC_L_BITS = [0, 2, 1, 3, 3, 2, 4, 3, 5, 5, 4, 4, 0, 0, 1, 0x7d]
_AC_L_VALS = [
    0x01, 0x02, 0x03, 0x00, 0x04, 0x11, 0x05, 0x12, 0x21, 0x31, 0x41, 0x06, 0x13, 0x51, 0x61, 0x07, 0x22, 0x71, 0x14, 0x32, 0x81, 0x91,
    0xa1, 0x08, 0x23, 0x42, 0xb1, 0xc1, 0x15, 0x52, 0xd1, 0xf0, 0x24, 0x33, 0x62, 0x72, 0x82, 0x09, 0x0a, 0x16, 0x17, 0x18, 0x19, 0x1a,
    0x25, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x34, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a, 0x53,
    0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78, 0x79,
    0x7a, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3, 0xa4, 0xa5,
    0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7, 0xc8, 0xc9,
    0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe1, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf1, 0xf2,
    0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa]
_AC_C_BITS = [0, 2, 1, 2, 4, 4, 3, 4, 7, 5, 4, 4, 0, 1, 2, 0x77]
_AC_C_VALS = [
    0x00, 0x01, 0x02, 0x03, 0x11, 0x04, 0x05, 0x21, 0x31, 0x06, 0x12, 0x41, 0x51, 0x07, 0x61, 0x71, 0x13, 0x22, 0x32, 0x81, 0x08, 0x14,
    0x42, 0x91, 0xa1, 0xb1, 0xc1, 0x09, 0x23, 0x33, 0x52, 0xf0, 0x15, 0x62, 0x72, 0xd1, 0x0a, 0x16, 0x24, 0x34, 0xe1, 0x25, 0xf1, 0x17,
    0x18, 0x19, 0x1a, 0x26, 0x27, 0x28, 0x29, 0x2a, 0x35, 0x36, 0x37, 0x38, 0x39, 0x3a, 0x43, 0x44, 0x45, 0x46, 0x47, 0x48, 0x49, 0x4a,
    0x53, 0x54, 0x55, 0x56, 0x57, 0x58, 0x59, 0x5a, 0x63, 0x64, 0x65, 0x66, 0x67, 0x68, 0x69, 0x6a, 0x73, 0x74, 0x75, 0x76, 0x77, 0x78,
    0x79, 0x7a, 0x82, 0x83, 0x84, 0x85, 0x86, 0x87, 0x88, 0x89, 0x8a, 0x92, 0x93, 0x94, 0x95, 0x96, 0x97, 0x98, 0x99, 0x9a, 0xa2, 0xa3,
    0xa4, 0xa5, 0xa6, 0xa7, 0xa8, 0xa9, 0xaa, 0xb2, 0xb3, 0xb4, 0xb5, 0xb6, 0xb7, 0xb8, 0xb9, 0xba, 0xc2, 0xc3, 0xc4, 0xc5, 0xc6, 0xc7,
    0xc8, 0xc9, 0xca, 0xd2, 0xd3, 0xd4, 0xd5, 0xd6, 0xd7, 0xd8, 0xd9, 0xda, 0xe2, 0xe3, 0xe4, 0xe5, 0xe6, 0xe7, 0xe8, 0xe9, 0xea, 0xf2,
    0xf3, 0xf4, 0xf5, 0xf6, 0xf7, 0xf8, 0xf9, 0xfa]


def _huff_codes(bits, vals):
    codes, code, k = {}, 0, 0
    for length in range(1, 17):
        for _ in range(bits[length - 1]):
            codes[vals[k]] = (code, length)
            code += 1
            k += 1
        code <<= 1
    return codes


class _BitSink:
    def __init__(self):
        self.out = bytearray()
        self.acc = 0
        self.n = 0

    def put(self, code, length):
        self.acc = (self.acc << length) | code
        self.n += length
        while self.n >= 8:
            b = (self.acc >> (self.n - 8)) & 0xFF
            self.out.append(b)
            if b == 0xFF:
                self.out.append(0)
            self.n -= 8
        self.acc &= (1 << self.n) - 1

    def flush(self):
        if self.n:
            self.put((1 << (8 - self.n)) - 1, 8 - self.n)


def _cat(v):
    a = abs(v)
    n = 0
    while a:
        n += 1
        a >>= 1
    return n


def _jpeg(rng, target):
    dcl, dcc = _huff_codes(_DC_L_BITS, _DC_VALS), _huff_codes(_DC_C_BITS, _DC_VALS)
    acl, acc = _huff_codes(_AC_L_BITS, _AC_L_VALS), _huff_codes(_AC_C_BITS, _AC_C_VALS)
    b = bytearray(b"\xff\xd8\xff\xe0\x00\x10JFIF\x00\x01\x01\x00\x00\x01\x00\x01\x00\x00")
    for t in range(2):
        b += b"\xff\xdb\x00\x43" + bytes([t]) + bytes(int(v) for v in np.clip(rng.integers(2, 60, size=64) + np.arange(64) // 2, 1, 255))
    b += b"\xff\xc0\x00\x11\x08\x01\xe0\x02\x80\x03\x01\x22\x00\x02\x11\x01\x03\x11\x01"
    for tc_th, bits, vals in ((0x00, _DC_L_BITS, _DC_VALS), (0x10, _AC_L_BITS, _AC_L_VALS), (0x01, _DC_C_BITS, _DC_VALS), (0x11, _AC_C_BITS, _AC_C_VALS)):
        b += b"\xff\xc4" + (3 + 16 + len(vals)).to_bytes(2, "big") + bytes([tc_th]) + bytes(bits) + bytes(vals)
    b += b"\xff\xda\x00\x0c\x03\x01\x00\x02\x11\x03\x11\x00\x3f\x00"
    sink = _BitSink()
    pred = [0, 0, 0]
    while len(b) + len(sink.out) < target - 16:
        for comp, nblk in ((0, 4), (1, 1), (2, 1)):          # 2x2 / 1x1 / 1x1 sampling: 6 blocks per MCU
            dct, act = (dcl, acl) if comp == 0 else (dcc, acc)
            for _ in range(nblk):
                dc = pred[comp] + int(rng.integers(-12, 13))
                dc = max(-1000, min(1000, dc))
                diff, pred[comp] = dc - pred[comp], dc
                s = _cat(diff)
                sink.put(*dct[s])
                if s:
                    sink.put(diff if diff > 0 else diff + (1 << s) - 1, s)
                run, k = 0, 1
                n_nz = int(rng.integers(1, 12))
                pos = np.sort(rng.choice(np.arange(1, 40), size=n_nz, replace=False))
                for p in pos:
                    run = int(p) - k
                    while run > 15:
                        sink.put(*act[0xF0])
                        run -= 16
                    v = int(rng.integers(1, 30 // (1 + int(p) // 6) + 2)) * (1 if rng.random() < 0.5 else -1)
                    s = _cat(v)
                    sink.put(*act[(run << 4) | s])
                    sink.put(v if v > 0 else v + (1 << s) - 1, s)
                    k = int(p) + 1
                sink.put(*act[0x00])
    sink.flush()
    b += sink.out
    return bytes(b[:target - 2]) + b"\xff\xd9"


def synth_binary(n_bytes, seed=0xE9E80003):
    """Alternating 64 KiB blocks: x86-64-ELF-like opcode streams and baseline-JPEG files."""
    rng = np.random.default_rng(seed)
    out = bytearray()
    opcodes = rng.integers(0, 256, size=256, dtype=np.uint8)
    weights = rng.dirichlet(np.full(256, 0.3))
    blk = 0
    while len(out) < n_bytes:
        if blk % 2 == 0:
            b = bytearray(b"\x7fELF\x02\x01\x01" + bytes(9) + b"\x02\x00\x3e\x00\x01\x00\x00\x00" + bytes(40))
            targets = rng.integers(0, 1 << 16, size=32)
            while len(b) < 65536:
                run = rng.choice(opcodes, size=int(rng.integers(8, 40)), p=weights)
                b += bytes(run)
                tgt = int(targets[rng.integers(32)]) - (len(b) & 0xFFFF)
                r = rng.random()
                op = b"\xe8" if r < 0.6 else (b"\xe9" if r < 0.85 else bytes([0x0F, 0x80 + int(rng.integers(16))]))
                b += op + int(tgt & 0xFFFFFFFF).to_bytes(4, "little")
            out += b[:65536]
        else:
            out += _jpeg(rng, 65536)
        blk += 1
    return bytes(out[:n_bytes])


if __name__ == "__main__":
    kind, n, path = sys.argv[1], int(sys.argv[2]), sys.argv[3]
    seed = int(sys.argv[4], 0) if len(sys.argv) > 4 else None
    fn = synth_text if kind == "text" else synth_binary
    data = fn(n, seed) if seed is not None else fn(n)
    open(path, "wb").write(data)
