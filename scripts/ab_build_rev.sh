#!/bin/bash
# Build the library as of git revision REV into multi-view-registration_b200/variants/lib_NAME.so (same-box A/B against the working tree):
#   scripts/ab_build_rev.sh REV NAME
set -e
REV=$1; NAME=$2
TMP=$(mktemp -d)
git archive $REV multi-view-registration_b200 include | tar -x -C $TMP
mkdir -p multi-view-registration_b200/variants
OUT=$PWD/multi-view-registration_b200/variants/lib_$NAME.so
(cd $TMP && python -c "
import sys; sys.path.insert(0, 'multi-view-registration_b200'); import build
print(build.build(force=True, out='$OUT'))")
rm -rf $TMP
