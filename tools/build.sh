#!/bin/bash
# Build the release library; exits non-zero on any compile error.
set -e
cd "$(dirname "$0")/../robust_e2e_gan_b200/csrc"
make -j8 > /tmp/re2e_make.log 2>&1 || { grep -E "error" /tmp/re2e_make.log *.ptxas.log | head -20; exit 1; }
grep -A2 "attloc_loop_.*ILi5ELi10ELi\(5\|10\)EEE" attloc_loop.ptxas.log | grep -E "spill|registers" || true
echo BUILD_OK
