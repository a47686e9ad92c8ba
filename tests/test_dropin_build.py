"""Drop-in boundary acceptance (SURVEY §7 step 3): the reference's own translation units —
src/main.cpp, xdr_server.cpp, audio_output.cpp, rtl_tcp_client.cpp, rtl_sdr_device.cpp,
config.cpp, signal_level.cpp, cpu_features.cpp — compile UNMODIFIED against the drop-in
headers (no liquid/liquid.h), and the whole application links against the engine libraries.
The build needs the reference's sources (FMTUNER_REFERENCE); the header check needs nothing."""
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import build_reference_app as bra  # noqa: E402


def test_dropin_headers_do_not_need_liquid():
    for dirpath, _, files in os.walk(os.path.join(ROOT, "fmtuner_sdr_b200", "dropin")):
        for f in files:
            for line in open(os.path.join(dirpath, f)):
                if line.lstrip().startswith("#"):
                    assert "liquid/liquid.h" not in line


@pytest.mark.skipif(not os.path.isdir(os.path.join(bra.REF, "src")), reason="reference sources not present")
def test_reference_application_builds_and_starts():
    from fmtuner_sdr_b200 import build as fmbuild
    fmbuild.build_lib()
    fmbuild.build_dropin()
    exe = bra.build()
    assert exe and os.path.exists(exe)
    out = subprocess.run([exe, "--help"], capture_output=True, text=True, timeout=60)
    assert "Usage:" in out.stdout and "--iq-rate" in out.stdout
    # the six DSP headers resolved to the drop-ins: no liquid symbol is referenced
    nm = subprocess.run(["nm", "-u", exe], capture_output=True, text=True).stdout
    assert "firfilt_crcf" not in nm and "nco_crcf" not in nm
