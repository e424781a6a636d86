#!/bin/bash
# Builds the CUDA library and fails loudly if anything goes wrong (so a stale .so is never sent to the GPU box).
set -e
out=$(make -C "$(dirname "$0")/../raytracing_rb_b200/csrc" -j4 2>&1) || { echo "$out" | grep -E "error|Stop" | head; echo BUILD FAILED; exit 1; }
echo "$out" | grep -E "error" && { echo BUILD FAILED; exit 1; }
echo BUILD OK
