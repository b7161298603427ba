#!/bin/sh
# Installs the UNMODIFIED reference package (peijin94/raytracingGRFF) into baseline/_ref (git-ignored), where
# bench.py's extras.reference_numpy leg and tests/test_bench_cli.py look for it:
#     sh baseline/install_ref.sh <path to a raytracingGRFF source checkout>
# The build writes an egg-info into the source tree: install from a temporary copy, so that a read-only checkout works.
# --no-deps: the only dependency is numpy, which the package's users already have.
set -e
src=${1:?usage: sh baseline/install_ref.sh <path to a raytracingGRFF source checkout>}
tmp=$(mktemp -d)
trap 'rm -rf "$tmp"' EXIT
cp -r "$src" "$tmp/ref"
chmod -R u+w "$tmp/ref"
python -m pip install --no-index --no-build-isolation --no-deps --target "$(dirname "$0")/_ref" --upgrade "$tmp/ref"
