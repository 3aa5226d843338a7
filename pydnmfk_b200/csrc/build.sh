#!/usr/bin/env bash
# Build libdnmf.so in-tree for sm_100a (nvcc cross-compiles without a GPU).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
OUT="${HERE}/../libdnmf.so"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
FLAGS=(-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC)
SRCS=(dnmf_core dnmf_api dnmf_bcd dnmf_comm dnmf_nmfk dnmf_resident dnmf_tc dnmf_tc_kl dnmf_tc_kl64 inst_row_f32 inst_row_f64 inst_col_f32 inst_col_f64 inst_small_f32 inst_small_f64 inst_row_a16 inst_col_a16 dnmf_tc16)
mkdir -p "${HERE}/build"
pids=()
objs=()
for f in "${SRCS[@]}"; do
  src="${HERE}/${f}.cu"; obj="${HERE}/build/${f}.o"
  objs+=("${obj}")
  # rebuild only when a source or header is newer than the object
  if [[ ! -f "${obj}" ]] || [[ -n "$(find "${HERE}" -maxdepth 1 \( -name '*.cuh' -o -name "${f}.cu" \) -newer "${obj}" -print -quit)" ]] \
     || [[ "${HERE}/../../include/dnmf.h" -nt "${obj}" ]]; then
    "${NVCC}" "${FLAGS[@]}" ${DNMF_PTXAS_V:+-Xptxas -v} -c -o "${obj}" "${src}" &
    pids+=($!)
  fi
done
for p in "${pids[@]:-}"; do [[ -n "${p}" ]] && wait "${p}"; done
"${NVCC}" -gencode arch=compute_100a,code=sm_100a -shared -o "${OUT}" "${objs[@]}" -lcudart_static -ldl -lpthread -lrt
echo "built ${OUT}"
