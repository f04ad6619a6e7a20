#!/bin/bash
# Regenerates tests/golden/generated.9.6 and generated.11.3 with the reference's own writer (tools/generateMatrix.cpp,
# built by `make -C oracle ref`); usage: REF=<checkout of the reference project> tests/golden/make_generated.sh.
# The tool seeds rand() with time(NULL), so every run gives different values; the committed files are one such run
# each and the tests only rely on the format and on round-tripping its values.
set -e
make -s -C "$(dirname "$0")/../../oracle" ref
"$(dirname "$0")/../../oracle/_ref/generateMatrix" 9 6 > "$(dirname "$0")/generated.9.6"
"$(dirname "$0")/../../oracle/_ref/generateMatrix" 11 3 > "$(dirname "$0")/generated.11.3"
