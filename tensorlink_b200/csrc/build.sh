#!/usr/bin/env bash
# Build libtensorlink_b200.so in-tree for sm_100a (the .so travels to the GPU box with the snapshot).
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
out="$here/libtensorlink_b200.so"
srcs=("$here"/*.cu)
hdrs=("$here"/*.cuh "$here/../../include/tensorlink_b200.h")
objs=()
mkdir -p "$here/build"
pids=()
stale() {  # object $1 of source $2: missing, or older than the source or any header
  [[ -f "$1" && ! "$2" -nt "$1" ]] || return 0
  for h in "${hdrs[@]}"; do [[ "$h" -nt "$1" ]] && return 0; done
  return 1
}
for s in "${srcs[@]}"; do
  o="$here/build/$(basename "${s%.cu}").o"
  objs+=("$o")
  if stale "$o" "$s"; then
    nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC \
         ${TL_NVCC_EXTRA:-} -c "$s" -o "$o" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [[ -n "$p" ]] && wait "$p"; done
nvcc -shared -o "$out" "${objs[@]}" -lcudart
echo "built $out"
