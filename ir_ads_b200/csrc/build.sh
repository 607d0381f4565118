#!/usr/bin/env bash
# Builds ir_ads_b200/libmsda_b200.so (the C-ABI library of include/msda.h) for sm_100a, in tree.
# nvcc cross-compiles without a GPU; the .so is git-ignored but ships to the GPU box with gpurun.
# One translation unit per kernel family (msda_host.h), compiled in parallel and only when one of its
# sources is newer than the object.  EXTRA_NVCC_FLAGS / OUT / OBJ_DIR serve tools/build_variant.sh.
set -euo pipefail
here="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
out="${OUT:-${here}/../libmsda_b200.so}"
obj="${OBJ_DIR:-${here}/../../build/obj}"
mkdir -p "${obj}"
FLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xptxas -v -Xcompiler -fPIC ${EXTRA_NVCC_FLAGS:-}"
hdrs="${here}/msda_coords.cuh ${here}/msda_scalar.cuh ${here}/msda_fast.cuh ${here}/msda_host.h ${here}/msda_fast_launch.cuh ${here}/../../include/msda.h"
compile() {   # compile <name> <extra deps...>
  local name="$1"; shift
  local src="${here}/${name}.cu" o="${obj}/${name}.o" stale=0
  for f in "${src}" ${hdrs} "$@" "${BASH_SOURCE[0]}"; do
    if [[ ! -f "${o}" || "${f}" -nt "${o}" ]]; then stale=1; fi
  done
  if [[ ${stale} == 1 ]]; then
    "${NVCC}" ${FLAGS} -c -o "${o}" "${src}" > "${obj}/build_${name}.log" 2>&1 || { cat "${obj}/build_${name}.log"; return 1; }
  fi
}
pids=()
compile msda_capi "${here}/msda_generic.cuh" "${here}/msda_det.cuh" & pids+=($!)
compile msda_fwd & pids+=($!)
compile msda_bwd & pids+=($!)
compile msda_bwd_aux & pids+=($!)
compile msda_fold "${here}/msda_fold.cuh" & pids+=($!)
compile msda_epilogue & pids+=($!)
compile msda_dcnv2 & pids+=($!)
rc=0
for p in "${pids[@]}"; do wait "${p}" || rc=1; done
[[ ${rc} == 0 ]] || { echo "build failed"; exit 1; }
"${NVCC}" -gencode arch=compute_100a,code=sm_100a -shared -o "${out}" "${obj}"/msda_capi.o "${obj}"/msda_fwd.o \
  "${obj}"/msda_bwd.o "${obj}"/msda_bwd_aux.o "${obj}"/msda_fold.o "${obj}"/msda_epilogue.o "${obj}"/msda_dcnv2.o
cat "${obj}"/build_msda_*.log > "${obj}/build.log" 2>/dev/null || true
echo "built ${out}"
