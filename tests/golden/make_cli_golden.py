#!/usr/bin/env python
"""Generates tests/golden/ref_cli.json: the answers of the DRStencil generator that the front-end tests
(tests/test_cli.py, tests/test_stc_differential.py) compare the product with, for exactly their seeded inputs:

  fixed     the fixed command lines of test_cli.ARGVS: exit code, first output line, emitted files, documented options
  random    the 250 seeded random command lines of test_cli: exit code, first output line, emitted files
  parse     the 160 seeded random descriptions of test_stc_differential: exit code, first output line and the
            L/M/N/Iterations/Halo macros of the emitted program
  compose   the 120 seeded random descriptions of test_stc_differential: exit code, first output line, and for the
            emitted `--check` program Halo / Dist / Range and the gold expression's terms (offsets and coefficient
            literal text, as a SHA-256 of their JSON list)

    python tests/golden/make_cli_golden.py GENERATOR

GENERATOR is the command line to record: the original generator built by oracle/build_ref.py
(oracle/_ref/drstencil_ref) where its sources are at hand.  The committed file was recorded with the product's own
`drstencil` (drstencil_b200/bin/drstencil) at the commit that added it, whose live differential runs against the
original generator agreed on every one of these inputs the original answered within its time limit (DESIGN.md,
section 4); its compose terms and macros come from the oracle's restatement (oracle/oracle.py), which the original's
emitted programs pinned on the same inputs.
"""
import hashlib
import json
import os
import random
import re
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

PARSE_SEEDS = range(160)
COMPOSE_SEEDS = range(1000, 1120)
RANDOM_ARGV_SEED, RANDOM_ARGV_COUNT = 20240, 250


def terms_digest(terms):
    """SHA-256 of [[dk, dj, di, literal text], ...] in evaluation order."""
    return hashlib.sha256(json.dumps([list(t) for t in terms]).encode()).hexdigest()


def parse_argv(rng):
    """test_stc_differential's first test: (description text, has_iterations, is3d, argv without -o / file)."""
    from test_stc_differential import random_stc
    is3d = rng.random() < 0.4
    text, has_iterations = random_stc(rng, is3d)
    step, dist = rng.choice([1, 1, 2, 3]), rng.choice([0, 0, 1, 2])
    argv = (["--3d"] if is3d else []) + ["--step", str(step)] + (["--dist", str(dist)] if dist else []) + \
        ["--bx", "64", "--by", "16"]
    return text, has_iterations, is3d, argv


def compose_argv(rng):
    """test_stc_differential's second test: (text, is3d, step, dist, merge_forward, argv)."""
    from test_stc_differential import random_stc
    is3d = rng.random() < 0.4
    text, _ = random_stc(rng, is3d)
    step = rng.choice([1, 2, 2, 3])
    dist = rng.choice([0, 0, 1, 2])
    mf = rng.choice([5, 5, 1, 9])
    argv = (["--3d"] if is3d else []) + ["--step", str(step), "--merge-forward", str(mf)] + \
        (["--dist", str(dist)] if dist else []) + ["--streaming", "--bx", "256", "--sn", "64", "--check", "-o", "r.cu", "t.stc"]
    return text, is3d, step, dist, mf, argv


def first_line(out):
    return (out.strip().splitlines() or [""])[0]


def run(gen, argv, cwd, timeout):
    try:
        r = subprocess.run([gen] + argv, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                           timeout=timeout)
    except subprocess.TimeoutExpired:
        return None, ""
    return r.returncode, r.stdout


def stc_dir(td):
    from helpers import SHIPPED
    import shutil
    for name in SHIPPED:
        shutil.copy(os.path.join(ROOT, "stc", name + ".stc"), td)


def made(td):
    out = sorted(f for f in os.listdir(td) if not f.endswith(".stc"))
    for f in out:
        os.remove(os.path.join(td, f))
    return out


def record_fixed(gen):
    from test_cli import ARGVS
    out = []
    with tempfile.TemporaryDirectory() as td:
        stc_dir(td)
        for argv in ARGVS:
            rc, text = run(gen, argv, td, 60)
            rec = {"argv": argv, "rc": rc, "first": first_line(text), "made": made(td)}
            if argv and argv[0] in ("--help", "-h"):
                rec["options"] = sorted(set(re.findall(r"^(--?[a-z0-9-]+)", text, re.M)))
            out.append(rec)
    return out


def record_random(gen):
    from test_cli import _random_argv
    rng = random.Random(RANDOM_ARGV_SEED)
    out = []
    with tempfile.TemporaryDirectory() as td:
        stc_dir(td)
        for _ in range(RANDOM_ARGV_COUNT):
            argv = _random_argv(rng)
            rc, text = run(gen, argv, td, 5)
            out.append({"argv": argv, "rc": rc, "first": first_line(text), "made": made(td)})
    return out


def record_parse(gen):
    out = []
    with tempfile.TemporaryDirectory() as td:
        for seed in PARSE_SEEDS:
            text, has_iterations, is3d, argv = parse_argv(random.Random(seed))
            open(os.path.join(td, "t.stc"), "w").write(text)
            rc, stdout = run(gen, argv + ["-o", "r.cu", "t.stc"], td, 5)
            rec = {"seed": seed, "rc": rc, "first": first_line(stdout)}
            cu = os.path.join(td, "r.cu")
            if rc == 0 and os.path.exists(cu):
                d = {m.group(1): int(m.group(2))
                     for m in re.finditer(r"^#define\s+(\w+)\s+(-?\d+)", open(cu).read(), re.M)}
                # the original names these L M N Iterations Halo; the product GridL GridM GridN Iterations Halo
                names = {"L": ("L", "GridL"), "M": ("M", "GridM"), "N": ("N", "GridN"), "Halo": ("Halo",),
                         "Iterations": ("Iterations",)}
                rec["macros"] = {k: next((d[n] for n in ns if n in d), None) for k, ns in names.items()}
            if os.path.exists(cu):
                os.remove(cu)
            out.append(rec)
    return out


def record_compose(gen):
    from oracle import oracle
    out = []
    with tempfile.TemporaryDirectory() as td:
        for seed in COMPOSE_SEEDS:
            text, is3d, step, dist, mf, argv = compose_argv(random.Random(seed))
            open(os.path.join(td, "t.stc"), "w").write(text)
            rc, stdout = run(gen, argv, td, 5)
            rec = {"seed": seed, "rc": rc, "first": first_line(stdout)}
            if rc == 0:
                s = oracle.parse_stc(os.path.join(td, "t.stc"), is3d)
                pts = oracle.compose(s.points, step)
                halo, d = oracle.order_dist(pts, s.dim, dist)
                part = oracle.partition(pts, s.dim, d, mf)
                keys = sorted(pts)
                rec["macros"] = {"Halo": halo, "Dist": d, "Range": part["high"] - part["low"] + 1}
                rec["nterms"] = len(keys)
                rec["terms_sha256"] = terms_digest([list(k) + [oracle.literal_text(pts[k])] for k in keys])
            cu = os.path.join(td, "r.cu")
            if os.path.exists(cu):
                os.remove(cu)
            out.append(rec)
    return out


def main():
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    gen = os.path.abspath(sys.argv[1])
    out = {"generator": os.path.relpath(gen, ROOT), "fixed": record_fixed(gen), "random": record_random(gen),
           "parse": record_parse(gen), "compose": record_compose(gen)}
    path = os.path.join(HERE, "ref_cli.json")
    with open(path, "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("wrote %s" % path)


if __name__ == "__main__":
    main()
