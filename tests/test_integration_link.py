"""INTEGRATION.md, verified: the reference's own daemon (rtlsdr_ft8d.c) and ft8_lib's example decoder (decode_ft8.c), patched
exactly as INTEGRATION.md sections 1 and 2 describe (tools/patch_reference_daemon.py, in a temp directory), compile against
include/ft8b200.h NEXT TO the reference's own headers and link against libft8b200.so with the hot-path objects (decode.o, ldpc.o,
unpack.o, kiss_fft) left out.  Needs the reference's sources where oracle/Makefile's REF points; nothing of them is copied into the repository."""
import os
import subprocess
import sys

import pytest

from oracle.pyoracle import reference_dir

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = reference_dir()
LIBDIR = os.path.join(ROOT, "rtlsdr-ft8d_b200")

pytestmark = pytest.mark.skipif(not os.path.isdir(os.path.join(REF, "ft8_lib")), reason="the reference's sources are not present (oracle/Makefile REF)")


@pytest.fixture(scope="module")
def patched(tmp_path_factory, pkg):
    pkg.lib()
    sys.path.insert(0, ROOT)
    from tools.patch_reference_daemon import patch, patch_decode_ft8
    out = tmp_path_factory.mktemp("refpatch")
    patch(REF, str(out))
    patch_decode_ft8(REF, str(out))
    os.symlink(os.path.join(REF, "ft8_lib"), out / "ft8_lib")
    return out


def undefined_symbols(binary):
    return set(line.split()[-1] for line in subprocess.check_output(["nm", "-D", "--undefined-only", str(binary)], text=True).splitlines())


def cuda_device_present():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def test_patched_daemon_builds_and_links_against_the_library(patched):
    ft8 = os.path.join(REF, "ft8_lib", "ft8")
    exe = patched / "rtlsdr_ft8d"
    # the daemon keeps pack/encode (its self-test synthesises with them) + what those need; decode.c, ldpc.c, unpack.c and FFTW are gone.
    # -O0 so that no call is optimised away behind the stubbed librtlsdr (oracle/shims: rtlsdr_open() always fails).
    cmd = ["gcc", "-O0", "-std=gnu17", "-w", "-I", os.path.join(ROOT, "oracle", "shims"), "-I", os.path.join(ROOT, "include"), "-I", str(patched),
           "-o", str(exe), str(patched / "rtlsdr_ft8d.c")] + [os.path.join(ft8, f) for f in ("constants.c", "pack.c", "text.c", "crc.c", "encode.c")] + \
          ["-L", LIBDIR, "-lft8b200", "-Wl,-rpath," + LIBDIR, "-lpthread", "-lm"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    undef = undefined_symbols(exe)
    for sym in ("rtlsdr_callback", "initFFTW", "freeFFTW", "ft8_subsystem", "ft8b200_stream_flip", "ft8b200_stream_decode", "ft8b200_stream_fetch"):
        assert sym in undef, sym + " must come from libft8b200.so"
    for sym in ("ft8_find_sync", "ft8_decode", "bp_decode", "unpack77", "fftwf_execute"):
        assert sym not in undef
    run = subprocess.run([str(exe), "-f", "2m", "-c", "A1XYZ", "-l", "AB12cd", "-t"], cwd=str(patched), capture_output=True, text=True)
    if cuda_device_present():
        assert run.returncode == 0 and "Self-test SUCCESS!" in run.stdout and "K1JT" in run.stdout
    else:
        assert run.returncode != 0 and "no CPU fallback" in run.stderr and "SUCCESS" not in run.stdout


def test_patched_decode_ft8_builds_and_links_against_the_library(patched):
    lib = os.path.join(REF, "ft8_lib")
    exe = patched / "decode_ft8"
    cmd = ["gcc", "-O0", "-std=gnu17", "-w", "-I", lib, "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(patched / "decode_ft8_main.c")] + \
          [os.path.join(lib, f) for f in ("ft8/encode.c", "ft8/crc.c", "ft8/text.c", "ft8/constants.c", "common/wave.c")] + \
          ["-L", LIBDIR, "-lft8b200", "-Wl,-rpath," + LIBDIR, "-lm"]
    p = subprocess.run(cmd, capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
    undef = undefined_symbols(exe)
    for sym in ("monitor_init", "monitor_process", "ft8_find_sync", "ft8_decode"):
        assert sym in undef, sym + " must come from libft8b200.so"
    assert not [s for s in undef if s.startswith("kiss_")]
    wav = os.path.join(lib, "tests", "191111_110130.wav")
    run = subprocess.run([str(exe), wav], capture_output=True, text=True)
    if cuda_device_present():
        assert run.returncode == 0 and run.stdout.count("\n") >= 5
    else:
        assert run.returncode != 0 and "no CPU fallback" in run.stderr and "000000" not in run.stdout


def test_header_coexists_with_the_reference_headers(tmp_path):
    """ft8b200.h after the reference's headers in one translation unit: no redefinition, and the layouts are the reference's."""
    src = tmp_path / "both.c"
    src.write_text('''
#include <stddef.h>
#include <stdint.h>
#include <stdbool.h>
#include <stdio.h>
#include <time.h>
#include <pthread.h>
#include "rtlsdr_ft8d.h"   /* not self-contained: rtlsdr_ft8d.c includes the system headers first */
#include "ft8_lib/ft8/constants.h"
#include "ft8_lib/ft8/decode.h"
#define FT8B200_WITH_RTLSDR_FT8D_H
#include "ft8b200.h"
_Static_assert(sizeof(waterfall_t) == 40 && offsetof(waterfall_t, mag) == 24 && offsetof(waterfall_t, protocol) == 36, "waterfall_t");
_Static_assert(sizeof(candidate_t) == 8 && sizeof(message_t) == 28 && sizeof(decode_status_t) == 12, "ft8_lib structs");
_Static_assert(sizeof(struct decoder_results) == 28 && sizeof(struct decoder_options) == 24, "daemon structs");
_Static_assert(sizeof(monitor_t) == 104, "monitor_t");
int main(void) { return PROTO_FT8 == 1 ? 0 : 1; }
''')
    p = subprocess.run(["gcc", "-std=gnu17", "-w", "-fsyntax-only", "-I", REF, "-I", os.path.join(ROOT, "oracle", "shims"), "-I", os.path.join(ROOT, "include"), str(src)],
                       capture_output=True, text=True)
    assert p.returncode == 0, p.stderr
