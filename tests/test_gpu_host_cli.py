"""The C++ host (pipsort_b200/host -> pipsort_b200/lib/PIPSORT): same command line, same six output files.

Every golden case stores the files the UNMODIFIED reference wrote (tests/golden/make_golden.py); the host CLI in
front of the GPU engine must reproduce them byte for byte (6 significant digits), including the stochastic
shotgun search (seed 12345, identical sampling sequence) and the appended _log.txt."""
import os
import subprocess
import tempfile

import pytest

from conftest import GOLDEN, ROOT, golden, has_golden

pytestmark = pytest.mark.gpu

CASES = ["small_c1_p075", "small_c2_p025", "small_c2_p075", "small_c3_p075", "small_c3_p0", "small_c3_g005_t1_s3",
         "small_sss_c3_p075", "small_sss_c2_p025", "example_c1_p025", "example_c2_p025", "example_sss_c2_p025",
         "small_given_72x5", "small_given_mixed_p025", "example_given_mixed"]
MAPS = {"small_example": "eur_afr_small_test_snp_map", "example": "snp_map"}


def host_bin():
    from pipsort_b200 import build
    build.build_engine()
    p = build.build_host()
    assert p and os.path.exists(p)
    return p


@pytest.mark.parametrize("name", CASES)
def test_cli_reproduces_reference_files(name):
    if not has_golden(name):
        pytest.skip("golden not generated")
    g = golden(name)
    d = os.path.join(GOLDEN, g["dataset"])
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "o")
        cmd = [host_bin(), "-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", MAPS[g["dataset"]], "-n", g["sample_sizes"],
               "-o", out] + [os.path.join(GOLDEN, a[1:]) if a.startswith("@") else a for a in g["args"]]
        p = subprocess.run(cmd, cwd=d, capture_output=True, text=True)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        for flag in g["stdout_flags"]:
            assert flag in p.stdout
        for suf, want in g["files"].items():
            with open(f"{out}_{suf}.txt") as f:
                got = f.read()
            assert got == want, f"{name}: {suf} differs"


def test_cli_shipped_example_files():
    """run_example.sh of the reference: -c 2 -n 334324,6771 -p 0.25 against the six expected_* files it ships."""
    d = os.path.join(GOLDEN, "example")
    with tempfile.TemporaryDirectory() as tmp:
        out = os.path.join(tmp, "results")
        p = subprocess.run([host_bin(), "-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", "snp_map", "-n", "334324,6771", "-o", out,
                            "-c", "2", "-p", "0.25"], cwd=d, capture_output=True, text=True)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        for suf in ["study0_post", "study1_post", "study0_set", "study1_set", "nocausal", "shared_pips"]:
            with open(f"{out}_{suf}.txt") as f, open(os.path.join(d, f"expected_{suf}.txt")) as w:
                assert f.read() == w.read(), suf


def test_cli_flag_quirks(tmp_path):
    """-m falls through into -n (pipsort.cpp:128-132): with -n BEFORE -m the sample sizes are overwritten by the map
    path and the run dies with the reference's format error; missing required flags exit 1."""
    d = os.path.join(GOLDEN, "small_example")
    out = str(tmp_path / "o")
    p = subprocess.run([host_bin(), "-l", "ldfiles.txt", "-z", "zfiles.txt", "-n", "7000,7000", "-m",
                        "eur_afr_small_test_snp_map", "-o", out], cwd=d, capture_output=True, text=True)
    assert p.returncode == 1 and "sample size is not in the right format" in p.stdout
    p = subprocess.run([host_bin(), "-l", "ldfiles.txt"], cwd=d, capture_output=True, text=True)
    assert p.returncode == 1 and "are required" in p.stdout
    # -b with the wrong -d: "config file is not the expected size" (postcal.cpp:434-437); -d 0: pipsort.cpp:190-193
    base = [host_bin(), "-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", "eur_afr_small_test_snp_map", "-n", "7000,7000", "-o", out,
            "-b", os.path.join(GOLDEN, "test_optional_configs", "all_configs_int16")]
    p = subprocess.run(base + ["-d", "71", "-e", "5"], cwd=d, capture_output=True, text=True)
    assert p.returncode == 1 and "config file is not the expected size" in p.stdout
    p = subprocess.run(base + ["-d", "0", "-e", "5"], cwd=d, capture_output=True, text=True)
    assert p.returncode == 1 and "Number of configs must be greater than 0" in p.stdout


def test_cli_several_devices_one_process():
    """PIPSORT_DEVICES=0,1 (or 0,0 on a single-GPU box: two engines on one device exercise the same shard + merge path):
    the rank space / the explicit-configuration rows are split over the engines, the stores merged -- same six files."""
    import torch
    devs = "0,1" if torch.cuda.device_count() > 1 else "0,0"
    for name in ["example_c2_p025", "small_c3_p075", "example_given_mixed"]:
        g = golden(name)
        d = os.path.join(GOLDEN, g["dataset"])
        with tempfile.TemporaryDirectory() as tmp:
            out = os.path.join(tmp, "o")
            cmd = [host_bin(), "-l", "ldfiles.txt", "-z", "zfiles.txt", "-m", MAPS[g["dataset"]], "-n", g["sample_sizes"],
                   "-o", out] + [os.path.join(GOLDEN, a[1:]) if a.startswith("@") else a for a in g["args"]]
            p = subprocess.run(cmd, cwd=d, capture_output=True, text=True, env=dict(os.environ, PIPSORT_DEVICES=devs))
            assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
            for suf, want in g["files"].items():
                with open(f"{out}_{suf}.txt") as f:
                    assert f.read() == want, f"{name}: {suf} differs"


def test_cli_synthetic_locus_with_psd_iterations_matches_engine():
    """A 400-SNP/study synthetic locus written in the reference's file formats: the determinant of its LD underflows, so
    Model's PSD loop really iterates (util.cpp:204-221) -- on the GPU in both paths.  The C++ host (files -> GPU
    pre-processing -> engine -> six files) must print the numbers the Python path (raw_ld engine) computes."""
    import numpy as np
    import pipsort_b200 as P
    from pipsort_b200 import synth
    L = synth.make_locus(400, overlap=0.8, seed=77, round_ld=False)
    with tempfile.TemporaryDirectory() as tmp:
        ld, z, mp, ns = synth.write_files(L, os.path.join(tmp, "in"))
        out = os.path.join(tmp, "o")
        p = subprocess.run([host_bin(), "-l", ld, "-z", z, "-m", mp, "-n", ns, "-o", out, "-c", "2", "-p", "0.5"],
                           capture_output=True, text=True)
        assert p.returncode == 0, p.stdout[-2000:] + p.stderr[-2000:]
        assert "diagonal shift 0," not in p.stdout                       # the loop added something
        with P.Engine(L.num_snps, L.sigma, L.z, L.d, 0.0, L.snp_map, gamma=0.01, sharing_param=0.5, max_causal=2,
                      raw_ld=True) as e:
            r = e.compute_total_likelihood(2)
            assert e.prep_info(0)["add_diag"] > 0
        pips = r.pips()
        got = [float(line.split("\t")[1]) for line in open(out + "_study0_post.txt").read().splitlines()[1:]]
        # 6 printed digits; the two runs sum in different orders, and printing rounds to 6 significant digits (5e-6 relative)
        np.testing.assert_allclose(got, pips[:400], rtol=6e-6, atol=1e-300)
        nc = [float(x) for x in open(out + "_nocausal.txt").read().split()]
        np.testing.assert_allclose(nc, r.no_causal(), rtol=6e-6, atol=1e-300)
