#!/bin/bash
# Installs the UNMODIFIED reference into baseline/_ref (git-ignored) for bench.py's reference arm:
#   baseline/install_ref.sh <numbskull source checkout>
# The checkout may be read-only and setup.py writes an egg-info next to itself, hence the writable copy;
# `future` (install_requires) need not be installed, hence --no-deps -- the one name the
# reference imports from it is provided by baseline/shims/past/builtins.py.
set -e
[ -d "$1/numbskull" ] || { echo "usage: $0 <numbskull source checkout>"; exit 1; }
src=$(cd "$1" && pwd)
cd "$(dirname "$0")/.."
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
rm -rf baseline/_ref && cp -r "$src" "$tmp/numbskull" && chmod -R u+w "$tmp"
python -m pip install -q --no-index --no-build-isolation --no-deps --target baseline/_ref "$tmp/numbskull"
diff -r -x __pycache__ "$src/numbskull" baseline/_ref/numbskull && echo "baseline/_ref/numbskull identical to the reference"
