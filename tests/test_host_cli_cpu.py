"""CPU-side checks of the C++ host in front of the engine: flag parsing and input validation end the run before any
device work, with the reference's messages and exit codes (pipsort.cpp:90-216, model.h:86-144)."""
import os
import subprocess
import tempfile

import numpy as np

from conftest import GOLDEN


def host_bin():
    from pipsort_b200 import build
    build.build_engine()
    p = build.build_host()
    assert p and os.path.exists(p)
    return p


def run(args, cwd):
    return subprocess.run([host_bin()] + args, cwd=cwd, capture_output=True, text=True)


def test_required_flags_and_argless_flags():
    d = os.path.join(GOLDEN, "small_example")
    p = run(["-l", "ldfiles.txt"], d)
    assert p.returncode == 1 and "Error: -l, -z, -o, and -n are required" in p.stdout        # pipsort.cpp:184-187
    p = run(["-h"], d)
    assert p.returncode == 1                                                                   # pipsort.cpp:92-95: optarg == NULL


def test_m_falls_through_into_n(tmp_path):
    """-m sets the snp_map AND the sample-size string (missing break, pipsort.cpp:128-132): with -n before -m the sizes
    are overwritten by the map's path and read_sigma rejects them."""
    d = os.path.join(GOLDEN, "small_example")
    p = run(["-l", "ldfiles.txt", "-z", "zfiles.txt", "-n", "7000,7000", "-m", "eur_afr_small_test_snp_map", "-o",
             str(tmp_path / "o")], d)
    assert p.returncode == 1 and "sample size is not in the right format" in p.stdout


def test_explicit_configuration_flag_checks(tmp_path):
    d = os.path.join(GOLDEN, "small_example")
    base = ["-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", "eur_afr_small_test_snp_map", "-n", "7000,7000", "-o", str(tmp_path / "o"), "-b",
            os.path.join(GOLDEN, "test_optional_configs", "all_configs_int16")]
    p = run(base + ["-d", "0", "-e", "5"], d)
    assert p.returncode == 1 and "Number of configs must be greater than 0" in p.stdout        # pipsort.cpp:190-193


def test_ld_and_z_size_mismatch_is_the_reference_error():
    """model.h:98-103: N is sqrt(#LD values); a z file with another number of SNPs ends the run with the 'nans' hint."""
    with tempfile.TemporaryDirectory() as tmp:
        np.savetxt(os.path.join(tmp, "a.ld"), np.eye(3))
        np.savetxt(os.path.join(tmp, "b.ld"), np.eye(2))
        with open(os.path.join(tmp, "a.z"), "w") as f:
            f.write("rs1 1.0\nrs2 0.5\n")                     # 2 SNPs against a 3 x 3 LD matrix
        with open(os.path.join(tmp, "b.z"), "w") as f:
            f.write("rs1 1.0\nrs2 0.5\n")
        with open(os.path.join(tmp, "ld.txt"), "w") as f:
            f.write("a.ld\nb.ld\n")
        with open(os.path.join(tmp, "z.txt"), "w") as f:
            f.write("a.z\nb.z\n")
        with open(os.path.join(tmp, "map"), "w") as f:
            f.write("rs1,0,0\nrs2,1,1\n")
        p = run(["-l", "ld.txt", "-z", "z.txt", "-m", "map", "-n", "100,100", "-o", os.path.join(tmp, "o")], tmp)
        assert p.returncode == 1 and "Check LD file for nans" in p.stdout
