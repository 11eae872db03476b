#!/bin/bash
# Where do the warps of the inter kernel spend their cycles?  (variant build with -DE264_INTER_TIMING: make variants)
# Inter kernel alone, 32 streams in flight; cycles of all warps summed per part of a chunk.  $1: library directory.
cd "$(dirname "$0")/.."; D=${1:-$PWD/edge264_b200/variants/itiming}
env LD_LIBRARY_PATH=$D E264_LIB_DIR=$D E264B_DIAG=1 S=32 STEPS=2 E264B_REPLAY_ONLY=1 timeout -k 5 300 python tools/replay_ab.py 2>&1 | grep -E "inter kernel|total"
