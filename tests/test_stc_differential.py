"""Randomised differential test of the .stc front end against the reference generator's answers
(tests/golden/ref_cli.json, made by tests/golden/make_cli_golden.py): random descriptions (keys in any
order, unknown tokens such as the shipped "iteratioins" typo, duplicate keys and points, radius 1-3,
2D and 3D, assorted coefficient spellings) run through both command lines with random --step/--dist;
exit code, first output line and the L/M/N/Iterations/Halo macros of the emitted programs must agree
(drstencil_2d.hpp:48-97, drstencil.hpp:52-103 of the original)."""
import json
import os
import random
import re
import subprocess
import sys

import pytest

from helpers import ROOT

sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))

CLI = os.path.join(ROOT, "drstencil_b200", "bin", "drstencil")
with open(os.path.join(ROOT, "tests", "golden", "ref_cli.json")) as _f:
    GOLDEN = json.load(_f)


def random_stc(rng, is3d):
    r = rng.choice([1, 1, 2, 3])
    dim = 3 if is3d else 2
    # the largest positive slow-axis offset bounds every other offset (what Halo is derived from)
    pts = [tuple([r] + [0] * (dim - 1))]
    pts += [tuple(rng.randint(-r, r) for _ in range(dim)) for _ in range(rng.randint(2, 9))]
    if rng.random() < 0.7:
        pts.append(tuple([-r] + [0] * (dim - 1)))
    coef = lambda: rng.choice(["0.2", "0.1", "0.05", ".5", "1e-1", "2", "-0.1", "0.125", "0.3333333", "1.5e-2", "0.07", "3"])
    keys = []
    if is3d or rng.random() < 0.2:
        keys.append(("L", str(rng.choice([64, 96, 130]))))
    keys.append(("M", str(rng.choice([64, 128, 512, 1000]))))
    keys.append(("N", str(rng.choice([64, 128, 512, 1024]))))
    has_iterations = rng.random() < 0.9
    if has_iterations:
        keys.append(("iterations", str(rng.choice([2, 4, 6, 10]))))
    rng.shuffle(keys)
    lines = []
    for name, value in keys:
        lines.append("%s %s" % (name, value))
        if rng.random() < 0.15:
            lines.append("%s %s" % (rng.choice(["foo", "iteratioins", "#", "bar"]), rng.choice(["7", "x"])))
        if rng.random() < 0.1:
            lines.append("%s %s" % (name, value))
    text = "\n".join(lines) + "\nstencil\n"
    for p in pts:
        text += " ".join(map(str, p)) + " " + coef() + rng.choice(["\n", " ", "\t\n"])
    return text, has_iterations


def _defines(path):
    if not os.path.exists(path):
        return {}
    return {m.group(1): int(m.group(2)) for m in re.finditer(r"^#define\s+(\w+)\s+(-?\d+)", open(path).read(), re.M)}


def test_random_descriptions_parse_and_analyse_like_the_reference(built, tmp_path):
    from make_cli_golden import parse_argv
    compared = emitted = 0
    assert [r["seed"] for r in GOLDEN["parse"]] == list(range(160))
    for ref in GOLDEN["parse"]:
        seed = ref["seed"]
        text, has_iterations, is3d, argv = parse_argv(random.Random(seed))
        (tmp_path / "t.stc").write_text(text)
        if os.path.exists(tmp_path / "o.cu"):
            os.remove(tmp_path / "o.cu")
        ours = subprocess.run([CLI] + argv + ["-o", "o.cu", "t.stc"], cwd=tmp_path, stdout=subprocess.PIPE,
                              stderr=subprocess.STDOUT, text=True, timeout=60)
        if ref["rc"] is None:                # the reference timed out on this input
            continue
        compared += 1
        assert ours.returncode == ref["rc"], (seed, argv, text, ours.stdout, ref)
        assert ours.stdout.strip().splitlines()[:1] == ([ref["first"]] if ref["first"] else []), (seed, argv, text)
        if ref["rc"] != 0:
            continue
        emitted += 1
        mine = _defines(tmp_path / "o.cu")
        pairs = {"M": "GridM", "N": "GridN", "Halo": "Halo"}
        if is3d:
            pairs["L"] = "GridL"
        if has_iterations:                 # without the key the reference prints an uninitialised int
            pairs["Iterations"] = "Iterations"
        for r, o in pairs.items():
            assert ref["macros"][r] == mine.get(o), (seed, argv, r, ref["macros"][r], mine.get(o), text)
    assert compared >= 150 and emitted >= 60, (compared, emitted)


def test_random_descriptions_compose_like_the_reference(built, tmp_path):
    """The gold expression the reference emits (`--check`) for random descriptions and steps: term order,
    offsets and the 6-significant-digit coefficient literals, plus the Halo / Dist / Range macros -- against
    BOTH the oracle's restatement (oracle/oracle.py) and the product's C ABI (drs_stencil_compose / _terms /
    _term_text / _analyze).  Many-digit coefficients (0.3333333 composed three times) exercise the literal
    round trip (drstencil_2d.hpp:174,231-251 of the original)."""
    from make_cli_golden import compose_argv, terms_digest
    import drstencil_b200 as drs
    from oracle import oracle
    checked = 0
    assert [r["seed"] for r in GOLDEN["compose"]] == list(range(1000, 1120))
    for ref in GOLDEN["compose"]:
        seed = ref["seed"]
        text, is3d, step, dist, mf, _ = compose_argv(random.Random(seed))
        (tmp_path / "t.stc").write_text(text)
        if ref["rc"] is None:
            continue
        # oracle restatement
        s = oracle.parse_stc(str(tmp_path / "t.stc"), is3d)
        pts = oracle.compose(s.points, step)
        halo, d = oracle.order_dist(pts, s.dim, dist)
        part = oracle.partition(pts, s.dim, d, mf)
        # product
        st = drs.Stencil.from_file(str(tmp_path / "t.stc"), is3d).compose(step)
        if ref["rc"] == 1:
            assert "No data to reuse" in ref["first"] and part is None, (seed, text)
            with pytest.raises(drs.DrsError):
                st.analyze(dist, mf)
            continue
        if ref["rc"] != 0:
            continue                        # "Invalid configuration!" depends on the tile, not on the operator
        macros = ref["macros"]
        keys = sorted(pts)
        assert len(keys) == ref["nterms"], (seed, text)
        assert terms_digest([list(k) + [oracle.literal_text(pts[k])] for k in keys]) == ref["terms_sha256"], (seed, text)
        assert macros["Halo"] == halo and macros["Dist"] == d and macros["Range"] == part["high"] - part["low"] + 1, (seed, text)
        mine = st.terms()
        texts = st.term_texts()
        assert terms_digest([list(t[:3]) + [x] for t, x in zip(mine, texts)]) == ref["terms_sha256"], (seed, text)
        assert [t[3] for t in mine] == [float(x) for x in texts], (seed, text)
        a = st.analyze(dist, mf)
        assert (a["halo"], a["dist"], a["range"]) == (macros["Halo"], macros["Dist"], macros["Range"]), (seed, text)
        checked += 1
    assert checked >= 60, checked
