"""HWA = trunc(HWF / HWN) as k_scan's 8-bit accumulator lanes compute it (a multiply by a reciprocal from a 256-entry table,
hdp_b200/csrc/seams.h: scan_hwa_rcp), checked without a GPU against integer division for every pair of 8-bit values.  The 16-bit
lanes divide with `/`."""
import ctypes
import os
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_hwa_reciprocal_exact_for_every_8bit_pair(tmp_path):
    so = str(tmp_path / "libscan_hwa_host.so")
    subprocess.run(["g++", "-O2", "-std=c++17", "-Wall", "-shared", "-fPIC", "-I", os.path.join(ROOT, "hdp_b200", "csrc"),
                    os.path.join(ROOT, "tests", "scan_hwa_host.cpp"), "-o", so], check=True)
    L = ctypes.CDLL(so)
    L.scan_hwa_mismatches.restype = ctypes.c_int64
    bad = (ctypes.c_uint32 * 2)()
    n = L.scan_hwa_mismatches(bad)
    assert n == 0, "%d pairs differ, first f = %d, nn = %d" % (n, bad[0], bad[1])
