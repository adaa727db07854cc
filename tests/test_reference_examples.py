"""The reference's own example programs (src/examples/*.c of SparseX) and its API test program (test/src/sparsex_test.c)
compile UNCHANGED against include/sparsex/*.h and link against libsparsex_b200.so.  They are compiled from where they lie
in a SparseX source tree (REF below) into tests/_refex/ (git-ignored), and run on the GPU — the test program through the
reference's own test script (test/scripts/test-sparsex.sh.in with its two @...@ placeholders filled in: 13 option sets on
the bundled matrices, two inputs that must fail).  These programs are SparseX's own sources, not part of this
repository, and what they check is their exit status and output as they run against this library, so there is nothing
to store in their place: without the source tree the tests skip."""
import os
import subprocess

import pytest

from tests.conftest import ROOT

REF = "/root/reference/src/examples"
REF_TEST = "/root/reference/test"
OUT = os.path.join(ROOT, "tests", "_refex")
PROGRAMS = ["csr_example", "mmf_example", "advanced_example", "matrix_caching_example_p1", "matrix_caching_example_p2",
            "reordering_example"]


def build_examples():
    import sparsex_b200
    libdir = os.path.dirname(sparsex_b200.lib_path())
    os.makedirs(OUT, exist_ok=True)
    for prog in PROGRAMS:
        subprocess.check_call(["gcc", "-std=gnu99", "-O1", "-w", os.path.join(REF, prog + ".c"), "-I", os.path.join(ROOT, "include"),
                               "-L", libdir, "-lsparsex_b200", "-lm", "-Wl,-rpath," + libdir, "-o", os.path.join(OUT, prog)])


def build_test_program():
    """test/src/sparsex_test.c unchanged; its check_result() (the reference's needs its internals) comes from
    tests/ref_test_check.c, the one internal header CsxCheck.hpp includes from tests/refshim_test/.  The test script is the
    reference's with @abs_top_builddir@ / @abs_top_srcdir@ pointing at tests/_refex and tests/golden."""
    import sparsex_b200
    libdir = os.path.dirname(sparsex_b200.lib_path())
    os.makedirs(os.path.join(OUT, "test", "src"), exist_ok=True)
    exe = os.path.join(OUT, "test", "src", "test_sparsex")
    subprocess.check_call(["gcc", "-std=gnu99", "-O1", "-w", os.path.join(REF_TEST, "src", "sparsex_test.c"),
                           os.path.join(ROOT, "tests", "ref_test_check.c"), "-I", os.path.join(ROOT, "tests", "refshim_test"),
                           "-I", os.path.join(ROOT, "include"), "-L", libdir, "-lsparsex_b200", "-lm", "-Wl,-rpath," + libdir, "-o", exe])
    text = open(os.path.join(REF_TEST, "scripts", "test-sparsex.sh.in")).read()
    # relative to the repository root (the script is run from there): the paths hold on the GPU box too
    text = text.replace("@abs_top_builddir@", "tests/_refex").replace("@abs_top_srcdir@/test/matrices", "tests/golden/matrices")
    with open(os.path.join(OUT, "test-sparsex.sh"), "w") as f:
        f.write(text)
    os.chmod(os.path.join(OUT, "test-sparsex.sh"), 0o755)


def test_reference_examples_compile_unchanged():
    if not os.path.isdir(REF):
        pytest.skip("reference tree not present")
    build_examples()
    for prog in PROGRAMS:
        assert os.path.exists(os.path.join(OUT, prog))
    build_test_program()
    assert os.path.exists(os.path.join(OUT, "test", "src", "test_sparsex"))
    # without a GPU the program still goes through its argument handling and the MMF reader: the unsorted file must be
    # refused normally (test_mmf_unsorted of the reference's script)
    r = subprocess.run([os.path.join(OUT, "test", "src", "test_sparsex"), "tests/golden/matrices/demopatt.mtx.unsorted"],
                       cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert 0 < r.returncode < 128 and "not sorted" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("prog,args", [("csr_example", []), ("mmf_example", ["tests/golden/matrices/demopatt.mtx.sorted"]),
                                       ("advanced_example", ["tests/golden/matrices/demopatt.mtx.sorted"]),
                                       ("reordering_example", ["tests/golden/matrices/symmetric.mtx.sorted"])])
def test_reference_examples_run(prog, args):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    exe = os.path.join(OUT, prog)
    if not os.path.exists(exe):
        pytest.skip("tests/_refex was not built (the reference tree is only present in the build container)")
    out = subprocess.run([exe] + args, capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]


@pytest.mark.gpu
def test_reference_test_script():
    """The reference's test suite (test/scripts/test-sparsex.sh.in) driving its own test program against this library."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    script = os.path.join(OUT, "test-sparsex.sh")
    if not os.path.exists(script) or not os.path.exists(os.path.join(OUT, "test", "src", "test_sparsex")):
        pytest.skip("tests/_refex was not built (the reference tree is only present in the build container)")
    out = subprocess.run(["bash", script], capture_output=True, text=True, timeout=900, cwd=ROOT)
    log = ""
    for name in ("test_sparsex.out", "test_sparsex.err"):
        path = os.path.join(ROOT, name)
        if os.path.exists(path):
            log += open(path).read()[-3000:]
            os.remove(path)
    assert "All tests passed!" in out.stdout and "FAILED" not in out.stdout, out.stdout + out.stderr + log
    assert out.stdout.count("PASSED") >= 13, out.stdout   # (the two must-fail inputs print PASSED only when the program exits non-zero)
