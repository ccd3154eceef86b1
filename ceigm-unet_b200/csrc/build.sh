#!/usr/bin/env bash
# Builds libss2d_b200.so in-tree for sm_100a (the only target). Usage: csrc/build.sh [extra nvcc flags]
# Every .cu is compiled to an object in parallel (objects are cached under csrc/build/ and rebuilt when the source
# or any header is newer), then linked into one shared library.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
ROOT="$(cd "$HERE/../.." && pwd)"
OUT="$HERE/../libss2d_b200.so"
OBJ="$HERE/build"
LOG="$HERE/../build_ptxas.log"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-std=c++17 -O3 -gencode arch=compute_100a,code=sm_100a -lineinfo --use_fast_math
       -Xcompiler -fPIC -I"$ROOT/include" -I"$HERE" -Xptxas -v "$@")
mkdir -p "$OBJ"
: > "$LOG"
newest_hdr=$(ls -t "$HERE"/*.cuh "$HERE"/*.h "$ROOT"/include/*.h "$HERE/build.sh" | head -1)
pids=()
srcs=("$HERE"/*.cu)
for src in "${srcs[@]}"; do
  base="$(basename "$src" .cu)"
  obj="$OBJ/$base.o"
  if [[ ! -f "$obj" || "$src" -nt "$obj" || "$newest_hdr" -nt "$obj" || $# -gt 0 ]]; then
    ( "$NVCC" "${FLAGS[@]}" -c -o "$obj" "$src" > "$OBJ/$base.log" 2>&1 || { cat "$OBJ/$base.log" >&2; rm -f "$obj"; exit 1; } ) &
    pids+=($!)
  fi
done
fail=0
for p in "${pids[@]:-}"; do
  [[ -z "$p" ]] && continue
  wait "$p" || fail=1
done
[[ $fail -eq 0 ]] || { echo "compile failed" >&2; exit 1; }
for src in "${srcs[@]}"; do
  base="$(basename "$src" .cu)"
  [[ -f "$OBJ/$base.log" ]] && { echo "==== $base.cu" >> "$LOG"; cat "$OBJ/$base.log" >> "$LOG"; }
done
objs=()
for src in "${srcs[@]}"; do objs+=("$OBJ/$(basename "$src" .cu).o"); done
"$NVCC" -shared -gencode arch=compute_100a,code=sm_100a -o "$OUT" "${objs[@]}"
echo "built $OUT"
