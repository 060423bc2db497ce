"""The audio-to-words Decoder's own code (file loading, argument plumbing, table sizing and retry, hypothesis and
segment extraction) on the CPU: device stages served by the compiled reference (front end, scorer, phone loop) and by
the host emulation of the search kernels (tools/dryrun/).  It must reproduce plain reference decodes -- words, path
score, every segment -- for the reference's test utterance and for one long stream at the beams of BASELINE config 5."""
import os
import subprocess
import sys

import pytest

from conftest import ROOT
from oracle import refdrv

pytestmark = pytest.mark.skipif(not refdrv.available(), reason="oracle/_ref/libpsref.so not built")


@pytest.fixture(scope="module")
def emul_libs(tmp_path_factory):
    from oracle import oracle
    oracle.build()
    d = str(tmp_path_factory.mktemp("dryemul"))
    for h in ("fsg", "ngs", "ngf"):
        subprocess.check_call(["g++", "-O1", "-fPIC", "-shared", "-ffp-contract=off", "-o", os.path.join(d, "lib%semul.so" % h),
                               os.path.join(ROOT, "tests", "emul", "%s_emul.cpp" % h), "-L" + os.path.join(ROOT, "oracle", "_build"),
                               "-lpsoracle", "-Wl,-rpath," + os.path.join(ROOT, "oracle", "_build")])
    return d


def run(emul_dir, script, *args):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "dryrun", script), *args], capture_output=True, text=True,
                       timeout=900, cwd=ROOT, env=dict(os.environ, PSB_EMUL_DIR=emul_dir))
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
    return r.stdout + r.stderr


@pytest.mark.timeout(1200)
def test_decoder_reproduces_reference_decodes(emul_libs):
    out = run(emul_libs, "decoder_dry.py")
    assert out.count("segments == reference") == 2 and "'go forward ten meters'" in out


@pytest.mark.timeout(1200)
def test_long_stream_beam_sweep_equals_reference(emul_libs):
    out = run(emul_libs, "beam_dry.py", "6")
    assert out.count("same hyp True, same score True") == 3 and "beam dry run ok" in out
    assert "emul: error" not in out                                  # tables sized from the stream length: no overflow retry
