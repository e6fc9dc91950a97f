#!/bin/bash
# Installs the UNMODIFIED reference package into baseline/_ref (git-ignored), where `bench.py --impl reference`
# finds it, with pip from a copy of the read-only tree (--no-deps: torch etc. are already installed).
set -e
cd "$(dirname "$0")/.."
rm -rf /tmp/refcopy && cp -r /root/reference /tmp/refcopy
python -m pip install --no-index --no-build-isolation --no-deps --find-links /opt/wheelhouse --upgrade --target baseline/_ref /tmp/refcopy
ls baseline/_ref | head -30
