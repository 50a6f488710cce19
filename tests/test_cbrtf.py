"""The builder's cube root (include/idk_cbrtf.h), shared by the host mirror and the device builder: glibc's cbrtf,
which is not correctly rounded, restated so that neither side depends on the platform's libm."""
import ctypes
import os
import platform
import subprocess

import numpy as np
import pytest

from idkengine_b200 import host

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(REPO, "tests", "golden", "cbrtf_sample.npz")


def shared_cbrtf(x):
    x = np.ascontiguousarray(x, np.float32)
    out = np.empty_like(x)
    L = host.lib()
    L.idkhost_cbrtf.restype = None
    L.idkhost_cbrtf.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_uint64]
    L.idkhost_cbrtf(x.ctypes.data, out.ctypes.data, len(x))
    return out


def test_shared_cbrtf_matches_stored_glibc_bits():
    """Every 65537th bit pattern (65,536 inputs over the whole range, both signs) plus zeros, infinities, NaN and
    subnormals, against the bits glibc 2.39's cbrtf returned for them."""
    g = np.load(GOLDEN)
    bits = g["input_bits"]
    got = shared_cbrtf(bits.view(np.float32)).view(np.uint32)
    want = g["cbrtf_bits"]
    nan = np.isnan(want.view(np.float32))
    assert np.array_equal(np.isnan(got.view(np.float32)), nan)
    assert np.array_equal(got[~nan], want[~nan])


def _glibc_version():
    try:
        return platform.libc_ver()
    except Exception:
        return ("", "")


@pytest.mark.skipif(_glibc_version() != ("glibc", "2.39") or not os.path.exists("/usr/bin/gcc"), reason="needs glibc 2.39 and gcc")
def test_shared_cbrtf_equals_glibc_on_every_input(tmp_path):
    """All 2^32 inputs against the C library's own cbrtf, 8 threads (~20 s)."""
    src = tmp_path / "cbrt_all.c"
    src.write_text(r'''
#include <math.h>
#include <pthread.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include "idk_cbrtf.h"
static unsigned long long bad[8];
static void* run(void* p) {
    const uint64_t w = (uint64_t)(uintptr_t)p;
    for (uint64_t b = w; b < (1ull << 32); b += 8) {
        uint32_t u = (uint32_t)b, ua, uc; float x, a, c;
        memcpy(&x, &u, 4); a = cbrtf(x); c = idk_cbrtf(x);
        memcpy(&ua, &a, 4); memcpy(&uc, &c, 4);
        if (ua != uc && !(isnan(a) && isnan(c))) bad[w]++;
    }
    return 0;
}
int main(void) {
    pthread_t t[8];
    for (uintptr_t i = 0; i < 8; i++) pthread_create(&t[i], 0, run, (void*)i);
    unsigned long long n = 0;
    for (int i = 0; i < 8; i++) { pthread_join(t[i], 0); n += bad[i]; }
    printf("%llu\n", n);
    return 0;
}
''')
    exe = tmp_path / "cbrt_all"
    subprocess.run(["gcc", "-O2", "-ffp-contract=off", "-I", os.path.join(REPO, "include"), str(src), "-o", str(exe), "-lm", "-pthread"], check=True)
    assert subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.strip() == "0"
