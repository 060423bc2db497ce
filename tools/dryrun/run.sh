#!/bin/bash
# Dry run of the gated GPU tests of the search kernels (tests/test_gpu_zz_*.py) on the CPU: torch's
# .cuda() becomes the identity and HmmContext's search methods are served by the host emulation
# harnesses (tests/emul/), so that what the tests compute, slice and compare is checked before GPU
# minutes are spent on them.  Expected: everything passes except the two tests that need the real
# library (block scan self-test, error reporting of psb_fsg_batch_device).
set -e
ROOT=$(cd "$(dirname "$0")/../.." && pwd)
D=$(mktemp -d)
export PSB_ROOT="$ROOT" PSB_EMUL_DIR="$D"
python -c "from oracle import oracle; oracle.build()" 2>/dev/null || (cd "$ROOT" && python -c "from oracle import oracle; oracle.build()")
for h in fsg ngs ngf; do
    g++ -O1 -fPIC -shared -ffp-contract=off -o "$D/lib${h}emul.so" "$ROOT/tests/emul/${h}_emul.cpp" -L"$ROOT/oracle/_build" -lpsoracle -Wl,-rpath,"$ROOT/oracle/_build"
done
cp "$ROOT/tools/dryrun/conftest_dry.py" "$D/conftest.py"
for f in test_gpu_zz_fsg.py test_gpu_zz_ngram.py; do
    python - "$ROOT/tests/$f" "$D/$f" <<'P'
import re, sys
s = open(sys.argv[1]).read()
s = re.sub(r'@pytest.fixture\(scope="module"\)\ndef api\(\):\n(    .*\n)+', '', s)
s = s.replace("d_scr.data_ptr()", "d_scr.numpy().ctypes.data").replace("d_pen.data_ptr()", "d_pen.numpy().ctypes.data")
open(sys.argv[2], "w").write(s)
P
done
cd "$D" && python -m pytest -q -m gpu -p no:cacheprovider --rootdir "$D" . | tail -n 5
# the audio-to-words Decoder with the device stages served by the compiled reference and the emulation
python "$ROOT/tools/dryrun/decoder_dry.py" | tail -n 3
