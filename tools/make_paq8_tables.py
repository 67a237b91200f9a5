"""Regenerate / check the constant tables carried as hex strings in cmix_b200/csrc/paq8_host.h (build container only).

    python tools/make_paq8_tables.py            print name + hex of every table
    python tools/make_paq8_tables.py --check    compare with the strings in paq8_host.h (exit 1 on a difference)

The values are what the reference's own initialisers produce: a throw-away program is compiled in a temp directory from
the table definitions where they lie in /root/reference/src/models/paq8.cpp (nothing is copied into the repo)."""
import os, re, subprocess, sys, tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = "/root/reference/src/models/paq8.cpp"
DUMP = r'''
static void dump(const char* name, const U8* p, int n){ printf("%s ", name); for(int i=0;i<n;i++) printf("%02x", p[i]); printf("\n"); }
'''


def lines(a, b):
    return "".join(open(REF).readlines()[a - 1:b])


def build(src, tmp, name):
    path = os.path.join(tmp, name + ".cpp")
    open(path, "w").write(src)
    exe = os.path.join(tmp, name)
    subprocess.run(["g++", "-w", path, "-o", exe], check=True)
    return subprocess.run([exe], check=True, capture_output=True, text=True).stdout


def tables():
    with tempfile.TemporaryDirectory() as tmp:
        a = build("#include <stdio.h>\ntypedef unsigned char U8; typedef unsigned int U32;\n" + lines(6607, 7050) + DUMP +
                  'int main(){ dump("exe_t1", Table1, 256); dump("exe_t2", Table2, 256); dump("exe_t3_38", Table3_38, 256); dump("exe_t3_3a", Table3_3A, 256);'
                  ' dump("exe_tx", TableX, 32); dump("exe_c1", TypeOp1, 256); dump("exe_c2", TypeOp2, 256); dump("exe_c3_38", TypeOp3_38, 256);'
                  ' dump("exe_c3_3a", TypeOp3_3A, 256); dump("exe_cx", TypeOpX, 32); dump("exe_invalid64", InvalidX64Ops, 19); dump("exe_prefix64", X64Prefixes, 8); return 0; }\n', tmp, "t")
        b = build("#include <stdio.h>\ntypedef unsigned char U8;\n" + lines(277, 341) + lines(3042, 3069) + DUMP +
                  'int main(){ dump("state", &State_table[0][0], 1024); dump("ascii_group_c0", AsciiGroupC0, 254); dump("ascii_group", AsciiGroup, 128); return 0; }\n', tmp, "t2")
    return dict(l.split() for l in (a + b).splitlines())


def differences(t):
    """Names of the tables whose hex strings in paq8_host.h differ from `t` (name -> hex)."""
    src = open(os.path.join(ROOT, "cmix_b200", "csrc", "paq8_host.h")).read()
    bad = []
    for name, want in t.items():
        field = {"state": r"&T\.state\[0\]\[0\]"}.get(name, r"T\." + name)
        m = re.search(r"unhex\(" + field + r", \d+,(.*?)\);", src, re.S)
        got = "".join(re.findall(r'"(.*?)"', m.group(1))) if m else ""
        if got != want:
            bad.append(name)
    return bad


def main():
    t = tables()
    if "--check" not in sys.argv:
        for k, v in t.items():
            print(k, v)
        return 0
    bad = differences(t)
    for name in bad:
        print("table", name, "differs")
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
