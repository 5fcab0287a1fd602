#!/usr/bin/env bash
# Build the C-ABI shared library for sm_100a (in-tree; the .so travels to the GPU box).
set -euo pipefail
ROOT="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
PKG="$ROOT/goal-conditioned-rl-framework_b200"
OUT="$PKG/gcrl_b200/libgcrl_b200.so"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17
       -Xcompiler -fPIC -Xcompiler -Wall -I"$ROOT/include" -I"$PKG/csrc")
mkdir -p "$PKG/build"
objs=()
pids=()
for src in "$PKG"/csrc/*.cu; do
  obj="$PKG/build/$(basename "${src%.cu}").o"
  if [[ ! -f "$obj" || "$src" -nt "$obj" || "$PKG/csrc/common.cuh" -nt "$obj" || "$ROOT/include/gcrl_b200.h" -nt "$obj" || -n "$(find "$PKG/csrc" -name '*.cuh' -newer "$obj" 2>/dev/null)" ]]; then
    echo "nvcc $(basename "$src")"
    rm -f "$obj"
    "$NVCC" "${FLAGS[@]}" ${EXTRA_NVCC_FLAGS:-} -c "$src" -o "$obj" &
    pids+=($!)
  fi
  objs+=("$obj")
done
# a bare `wait` returns 0 whatever the jobs returned: wait on each, so that a failed compile stops the build
failed=0
for pid in "${pids[@]}"; do
  wait "$pid" || failed=1
done
(( failed == 0 )) || { echo "build.sh: compilation failed" >&2; exit 1; }
"$NVCC" -Wno-deprecated-gpu-targets -shared -o "$OUT" "${objs[@]}" -lcudart_static -lpthread -ldl -lrt
echo "built $OUT"
