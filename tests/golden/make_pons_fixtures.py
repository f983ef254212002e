"""Copies the reference's known-answer DATA files (not source code) for Connect-Four:
games/connect-four/benchmark/Test_L*_R* -- 6 x 1000 lines "moves score" with exact
solver scores (consumed by the reference at scripts/pons_benchmark.jl:49-78).
The tests only read the committed copies.
Usage:  python tests/golden/make_pons_fixtures.py <AlphaZero.jl checkout>"""
import hashlib, os, shutil, sys
SRC = os.path.join(sys.argv[1], "games", "connect-four", "benchmark")
DST = os.path.join(os.path.dirname(os.path.abspath(__file__)), "pons")
os.makedirs(DST, exist_ok=True)
with open(os.path.join(DST, "MD5SUMS"), "w") as f:
    for name in sorted(os.listdir(SRC)):
        shutil.copyfile(os.path.join(SRC, name), os.path.join(DST, name))
        f.write("%s  %s\n" % (hashlib.md5(open(os.path.join(SRC, name), "rb").read()).hexdigest(), name))
