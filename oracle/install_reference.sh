#!/bin/sh
# Recipe for the reference-as-shipped CPU arm (bench.py --impl reference, oracle/ref_arm.py) and for the reference's own test files
# (tests/test_gpu_reference_suite.py):  sh oracle/install_reference.sh [StochVolModels source tree]
# installs the UNMODIFIED upstream package (ArturSepp/StochVolModels 2.2.0) into git-ignored oracle/_ref.  The source tree is the
# argument, else $B200SV_REFERENCE_SRC, else /root/reference (the default location of the upstream checkout); without a readable tree there is
# nothing to install and the script exits 0.
# The wheel is built from a temporary copy so that the source tree may be read-only; --no-deps because matplotlib / seaborn /
# vanilla-option-pricers are not needed by the timed calls (oracle/ref_arm.py stubs them).
set -e
src="${1:-${B200SV_REFERENCE_SRC:-/root/reference}}"
if [ ! -r "$src/src/stochvolmodels/__init__.py" ]; then
    echo "install_reference.sh: no readable StochVolModels source tree at $src; oracle/_ref not installed"
    exit 0
fi
cd "$(dirname "$0")/.."
tmp="$(mktemp -d)"
trap 'rm -rf "$tmp"' EXIT
cp -r "$src" "$tmp/src"
chmod -R u+w "$tmp/src"
rm -rf oracle/_ref
"${PYTHON:-python}" -m pip install --no-index --no-build-isolation --no-deps --target oracle/_ref "$tmp/src"
