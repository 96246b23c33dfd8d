"""The `drstencil` command line against the original generator's answers (tests/golden/ref_cli.json, made by
tests/golden/make_cli_golden.py): same exit codes and messages for the same argv (CPU), and the emitted
program compiled with nvcc and run on the GPU (gpu)."""
import json
import os
import re
import shutil
import subprocess

import pytest

from helpers import ROOT, SHIPPED

CLI = os.path.join(ROOT, "drstencil_b200", "bin", "drstencil")
with open(os.path.join(ROOT, "tests", "golden", "ref_cli.json")) as _f:
    GOLDEN = json.load(_f)

ARGVS = [
    [],
    ["--help"],
    ["-h"],
    ["2d5pt_star.stc"],
    ["--step", "2d5pt_star.stc"],                 # valued option in the last-but-one slot
    ["--bx", "2d5pt_star.stc"],
    ["--merge-forward", "2d5pt_star.stc"],
    ["-o", "2d5pt_star.stc"],                     # silently ignored
    ["--frobnicate", "3", "2d5pt_star.stc"],      # unknown option
    ["missing.stc"],
    ["2d5pt_cross.stc"],                          # no data to reuse
    ["--dist", "2", "2d5pt_cross.stc"],
    ["--3d", "3d9pt_cross.stc"],
    ["--3d", "--dist", "2", "3d9pt_cross.stc"],
    ["--3d", "--step", "2", "3d7pt_star.stc"],
    ["--step", "2", "--bx", "4", "2d9pt_box.stc"],           # invalid configuration
    ["--3d", "--step", "2", "--by", "4", "--merge-forward", "1", "3d7pt_star.stc"],
    ["--step", "4", "--streaming", "--bx", "128", "--sn", "64", "--check", "-o", "x.cu", "2d9pt_box.stc"],
    ["--streaming", "--bx", "128", "--sn", "64", "--cyclic-merge-x", "2", "--prefetch", "--gold", "2d25pt_box.stc"],
    ["--step", "3", "2d5pt_cross.stc"],
    ["--step", "2", "--dist", "1", "2d9pt_cross.stc"],
]


def _run(binary, argv, cwd, timeout=60):
    try:
        r = subprocess.run([binary] + argv, cwd=cwd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True,
                           timeout=timeout)
    except subprocess.TimeoutExpired:
        return "timeout", ""
    return r.returncode, r.stdout


def test_exit_codes_and_messages_match_the_reference_binary(built, tmp_path):
    assert [r["argv"] for r in GOLDEN["fixed"]] == ARGVS
    for name in SHIPPED:
        shutil.copy(os.path.join(ROOT, "stc", name + ".stc"), tmp_path)
    for ref in GOLDEN["fixed"]:
        argv = ref["argv"]
        rc_o, out_o = _run(CLI, argv, tmp_path)
        assert rc_o == ref["rc"], (argv, rc_o, ref, out_o)
        if argv and argv[0] in ("--help", "-h"):
            for opt in ref["options"]:                                    # every reference option is documented
                assert opt in out_o, opt
            continue
        assert out_o.strip().splitlines()[:1] == ([ref["first"]] if ref["first"] else []), (argv, out_o, ref)
        # both write (or do not write) an output file
        made_o = sorted(f for f in os.listdir(tmp_path) if f.endswith(".cu"))
        assert made_o == [f for f in ref["made"] if f.endswith(".cu")], (argv, made_o, ref)
        for f in made_o:
            os.remove(tmp_path / f)


def test_emitted_program_is_self_contained_text(built, tmp_path):
    shutil.copy(os.path.join(ROOT, "stc", "2d9pt_box.stc"), tmp_path)
    rc, out = _run(CLI, ["--step", "2", "--check", "--dtype", "f32", "--info", "-o", "k.cu", "2d9pt_box.stc"], tmp_path)
    assert rc == 0 and "Halo 2 Dist 2 Range 3" in out
    text = open(tmp_path / "k.cu").read()
    for needle in ("#define DRS_T float", "#define DRS_TS 2", "drs_sweep2d.cuh", "gold_2d9pt_box", "Initiating ...",
                   "GPU computation time: %f ms", "[Test] RMS Error: %e", "#define Iterations 4"):
        assert needle in text, needle


def test_emitted_program_runs_every_sub_step_of_an_unfused_3d_temporal_sweep(built, tmp_path):
    """`--3d --step 5 --fuse temporal` is too deep for the fused kernel: one sweep = five single-step launches with
    frozen rings r, 2r, ... (KernelSpec::sub_launches).  The emitted program must do the same (round 1: it launched
    once per sweep, advanced one timestep instead of five and failed its own --check)."""
    shutil.copy(os.path.join(ROOT, "stc", "3d7pt_star.stc"), tmp_path)
    rc, out = _run(CLI, ["--3d", "--step", "5", "--fuse", "temporal", "--check", "-o", "x.cu", "3d7pt_star.stc"], tmp_path)
    assert rc == 0, out
    text = open(tmp_path / "x.cu").read()
    assert "#define Halo 5" in text and "#define Step 5" in text
    assert "for (int s = 1; s <= 5; ++s)" in text and "dr_launch_one(src, dst, s * 1);" in text
    assert "scratch[(s - 1) & 1]" in text
    # a fused (or single-step) program launches once per sweep
    rc, out = _run(CLI, ["--3d", "--step", "2", "--check", "-o", "y.cu", "3d7pt_star.stc"], tmp_path)
    assert rc == 0, out
    assert "dr_launch_one(in, out, Halo);" in open(tmp_path / "y.cu").read()


@pytest.mark.gpu
@pytest.mark.parametrize("argv,name,exact", [
    (["--check"], "2d5pt_star", True),
    (["--step", "2", "--check"], "2d9pt_box", False),
    (["--3d", "--check"], "3d7pt_star", True),
    (["--3d", "--step", "5", "--fuse", "temporal", "--check"], "3d7pt_star", False),
])
def test_emitted_program_builds_and_checks_out_on_gpu(built, tmp_path, argv, name, exact):
    """`drstencil ... -o out.cu` -> nvcc -> run: the reference's stdout protocol, error at the floor."""
    if shutil.which("nvcc") is None:
        pytest.skip("nvcc not on PATH")
    src = open(os.path.join(ROOT, "stc", name + ".stc")).read()
    src = re.sub(r"\b([LMN]) \d+", lambda m: m.group(1) + (" 96" if m.group(1) == "L" else " 328"), src)
    open(tmp_path / (name + ".stc"), "w").write(src)
    rc, out = _run(CLI, argv + ["-o", "out.cu", name + ".stc"], tmp_path)
    assert rc == 0, out
    r = subprocess.run(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-lineinfo",
                        "--fmad=false", "-I", os.path.join(ROOT, "drstencil_b200", "csrc", "kernels"), "out.cu", "-o", "out"],
                       cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert r.returncode == 0, r.stdout
    r = subprocess.run(["./out"], cwd=tmp_path, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True, timeout=120)
    assert r.returncode == 0, r.stdout
    lines = r.stdout.splitlines()
    assert lines[0] == "Initiating ..." and "GPU computing ..." in lines and "GPU finished computing." in lines
    assert any(l.startswith("GPU computation time: ") and l.endswith(" ms") for l in lines)
    mx = float(re.search(r"\[Test\] Max Error : (\S+)", r.stdout).group(1))
    rms = float(re.search(r"\[Test\] RMS Error: (\S+)", r.stdout).group(1))
    if exact:
        assert mx == 1e-13 and rms == 0.0        # bit-identical to the gold kernel
    else:
        assert mx < 1e-12


@pytest.mark.gpu
def test_cli_run_mode_on_gpu(built, tmp_path):
    src = open(os.path.join(ROOT, "stc", "2d9pt_box.stc")).read().replace("8192", "1024")
    open(tmp_path / "2d9pt_box.stc", "w").write(src)
    rc, out = _run(CLI, ["--step", "4", "--check", "--run", "2d9pt_box.stc"], tmp_path)
    assert rc == 0, out
    assert "GPU computation time:" in out and "[Test] RMS Error:" in out
    assert float(re.search(r"\[Test\] Max Error : (\S+)", out).group(1)) < 1e-12


_VALUED = ["--step", "--dist", "--bx", "--by", "--sn", "--stream-unroll", "--block-merge-x", "--block-merge-y",
           "--cyclic-merge-x", "--cyclic-merge-y", "--merge-forward"]
_FLAGS = ["--streaming", "--prefetch", "--check", "--gold", "--3d"]


def _random_argv(rng):
    """Random command lines from the reference's option grammar, including malformed ones (a valued option
    without its value, unknown options, `-o` with and without a file name, non-numeric and non-positive
    values).  Left out on purpose: `--step` < 1 (the reference segfaults) and a 3D description parsed without
    `--3d` (the reference never returns: its token loop spins on the fourth column, SURVEY 8a-1)."""
    argv = []
    for _ in range(rng.randint(0, 6)):
        k = rng.random()
        if k < 0.55:
            opt = rng.choice(_VALUED)
            val = rng.choice(["1", "2", "3", "4"] if opt == "--step" else
                             ["1", "2", "3", "4", "8", "16", "32", "64", "128", "0", "-1", "x", "256"])
            argv += [opt, val] if rng.random() < 0.93 else [opt]
        elif k < 0.85:
            argv.append(rng.choice(_FLAGS))
        elif k < 0.92:
            argv += ["-o", rng.choice(["out.cu", "k.cu"])] if rng.random() < 0.8 else ["-o"]
        else:
            argv.append(rng.choice(["--bogus", "-x", "--help", "-h", "foo"]))
    name = rng.choice(SHIPPED)
    if name.startswith("3d") and "--3d" not in argv:
        argv.insert(rng.randint(0, len(argv)), "--3d")
    if rng.random() < 0.95:
        argv.append(name + ".stc")
    return argv


def test_random_command_lines_against_the_reference_binary(built, tmp_path):
    """Differential test: 250 seeded random command lines give the same exit code, the same first line
    of output and the same set of emitted files as the reference binary."""
    import random
    for name in SHIPPED:
        shutil.copy(os.path.join(ROOT, "stc", name + ".stc"), tmp_path)
    rng = random.Random(20240)
    first = lambda s: (s.strip().splitlines() or [""])[0]
    hung_or_crashed = []
    assert len(GOLDEN["random"]) == 250
    for ref in GOLDEN["random"]:
        argv = _random_argv(rng)
        assert argv == ref["argv"]
        rc_o, out_o = _run(CLI, argv, tmp_path, timeout=20)
        made_o = sorted(f for f in os.listdir(tmp_path) if not f.endswith(".stc"))     # `-o --3d` names a file "--3d"
        for f in made_o:
            os.remove(tmp_path / f)
        assert rc_o != "timeout", argv
        if ref["rc"] is None or ref["rc"] < 0:
            hung_or_crashed.append(argv)         # the reference spins or dies on this input: nothing to compare
            continue
        assert rc_o == ref["rc"], (argv, rc_o, ref, out_o)
        assert made_o == ref["made"], (argv, made_o, ref)
        if not (argv and argv[0] in ("--help", "-h")):
            assert first(out_o) == ref["first"], (argv, out_o, ref)
    assert len(hung_or_crashed) <= 10, hung_or_crashed
