#!/bin/bash
# Builds libmgv_b200.so (C ABI, see include/mgv_b200.h) for sm_100a, in-tree.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${MGV_OUT:-${HERE}/../deepgate/_lib}"
mkdir -p "${OUT}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -O2 ${MGV_NVCC_EXTRA:-})
OBJS=()
pids=()
for f in mgv_error schedule sweep sweep_tc struct_tc struct_bwd_tc linear linear_tc vae_func recon readout pack tc_selftest logic_sim; do
  "${NVCC}" "${FLAGS[@]}" -c "${HERE}/${f}.cu" -o "${OUT}/${f}.o" &
  pids+=($!)
  OBJS+=("${OUT}/${f}.o")
done
for p in "${pids[@]}"; do wait "$p"; done
"${NVCC}" -shared -o "${OUT}/libmgv_b200.so" "${OBJS[@]}" -lcudart
echo "built ${OUT}/libmgv_b200.so"
