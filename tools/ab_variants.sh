#!/bin/bash
# Same-box A/B of kernel build variants (run it inside ONE gpurun call: GPUs of the pool differ by ~10 %).
#   tools/ab_variants.sh build "-DSOME_FLAG" "-DSOME_FLAG -DOTHER_FLAG" ...    # here: cross-compile one .so per flag set
#   gpurun -- 'tools/ab_variants.sh run'                                       # on the GPU box: parity + timings per variant
# Variant 0 is always the product build (no extra flags).
set -e
ROOT="$(cd "$(dirname "$0")/.." && pwd)"
SRC="$ROOT/peaksegdisk_b200/csrc"
OUT="$ROOT/peaksegdisk_b200"
NVFLAGS="-gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -fmad=false -Xcompiler -fPIC,-ffp-contract=off,-Wno-unused-function -shared"
case "$1" in
build)
  shift
  rm -f "$OUT"/libpsd_ab*.so "$OUT"/libpsd_ab.txt
  k=1
  for flags in "$@"; do
    echo "variant $k: $flags" | tee -a "$OUT/libpsd_ab.txt"
    (cd "$SRC" && /usr/local/cuda/bin/nvcc ${NVFLAGS% -shared} $flags -DPSD_G32 -c -o "/tmp/psd_ab_lat$k.o" fpop_lat.cu &&
      /usr/local/cuda/bin/nvcc $NVFLAGS $flags -Xptxas -v -o "$OUT/libpsd_ab$k.so" fpop_gpu.cu host_api.cpp "/tmp/psd_ab_lat$k.o" 2>&1 | grep -A2 "fpop_dp_kernelILi16ELi1E" | grep -E "spill|Used" | head -2)
    k=$((k + 1))
  done
  ;;
run)
  cd "$ROOT"
  cat "$OUT/libpsd_ab.txt" 2>/dev/null || true
  for lib in "$OUT/libpeaksegdisk_b200.so" "$OUT"/libpsd_ab*.so; do
    echo "== $(basename "$lib")"
    export PSD_LIB="$lib"
    python -m pytest tests/test_gpu_parity.py -m gpu -q -x -k "golden or fresh_seeds or synthetic or fuzz or full_size" 2>&1 | tail -1
    PSD_OCCUPANCY_MODE=1 python tools/prof_case.py 1600 3000 2 | tail -1
    PSD_LATENCY_MODE=1 python tools/prof_case.py 29 20000 2 | tail -1
    python bench.py --steps 1 --warmup 3 --no-cpu-baseline | python -c "
import json,sys
d=json.loads(sys.stdin.read().strip().splitlines()[-1]); print('config 2: value %.4g  e2e %.4g  ms/step %.1f' % (d['value'], d['e2e']['value'], d['ms_per_step']))"
  done
  ;;
*)
  echo "usage: $0 build <flags>... | run"; exit 2;;
esac
