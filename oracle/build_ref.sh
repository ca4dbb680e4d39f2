#!/usr/bin/env bash
# Compiles the UNMODIFIED reference (facebookresearch/dietgpu) CUDA + host
# sources, from where they lie under $REF (default /root/reference), for
# sm_100a into oracle/_ref/libdietgpu_ref.so, together with oracle/ref_harness.cu
# (a C-ABI veneer written for this repo) and the glog stand-in in
# oracle/ref_shim/.  Drives nvcc directly -- the reference's own CMake build
# is NOT run.  Outputs only into oracle/_ref/ (git-ignored, travels to the GPU
# box with gpurun).  TEST / BASELINE infrastructure only.
#
# `build_ref.sh gtests` instead compiles the reference's own googletest suites
# (ans/ANSTest.cu, float/FloatTest.cu), unchanged, into oracle/_ref/ref_ans_test
# and ref_float_test, run by tests/test_gpu_reference_gtests.py.  Unlike the
# rest of oracle/_ref/, these binaries depend on this project: they compile
# include/dietgpu_b200_compat.hpp (through the include-path shim tests/ref_shim)
# and link dietgpu_b200/libdietgpu_b200.so, which must be built first.  Wherever
# the reference's sources exist they are deleted and rebuilt, and build() fails
# if they do not compile; elsewhere binaries from an earlier build are kept.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${REF:-/root/reference}"
OUT="$HERE/_ref"
if [ ! -d "$REF/dietgpu" ]; then
  echo "build_ref: $REF/dietgpu not present; keeping any prebuilt $OUT" >&2
  exit 0
fi
mkdir -p "$OUT/obj"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
if [ "${1:-}" = gtests ]; then
  ROOT="$(cd "$HERE/.." && pwd)"
  GT="$REF/third_party/googletest/googletest"
  rm -f "$OUT/ref_ans_test" "$OUT/ref_float_test"
  mkdir -p "$OUT/gtest"
  if [ ! -f "$OUT/gtest/gtest-all.o" ]; then
    g++ -std=c++17 -O1 -I"$GT/include" -I"$GT" -c "$GT/src/gtest-all.cc" -o "$OUT/gtest/gtest-all.o"
    g++ -std=c++17 -O1 -I"$GT/include" -I"$GT" -c "$GT/src/gtest_main.cc" -o "$OUT/gtest/gtest_main.o"
  fi
  GFLAGS=(-std=c++17 -O2 -gencode arch=compute_100a,code=sm_100a -ccbin /usr/bin/g++
          -I"$ROOT/tests/ref_shim" -I"$ROOT/include" -I"$GT/include")
  GLINK=(-L"$ROOT/dietgpu_b200" -ldietgpu_b200 -Xlinker -rpath -Xlinker '$ORIGIN/../../dietgpu_b200' -lcudart -lpthread)
  "$NVCC" "${GFLAGS[@]}" -o "$OUT/ref_ans_test" "$REF/dietgpu/ans/ANSTest.cu" "$OUT"/gtest/*.o "${GLINK[@]}"
  "$NVCC" "${GFLAGS[@]}" -o "$OUT/ref_float_test" "$REF/dietgpu/float/FloatTest.cu" "$OUT"/gtest/*.o "${GLINK[@]}"
  echo "built $OUT/ref_ans_test $OUT/ref_float_test"
  exit 0
fi
FLAGS=(-std=c++17 -O2 -DNDEBUG -gencode arch=compute_100a,code=sm_100a -lineinfo
       -I"$REF" -I"$HERE/ref_shim" -Xcompiler -fPIC -ccbin /usr/bin/g++ -w)
SRCS=(dietgpu/ans/GpuANSEncode.cu dietgpu/ans/GpuANSDecode.cu dietgpu/ans/GpuANSInfo.cu
      dietgpu/float/GpuFloatCompress.cu dietgpu/float/GpuFloatDecompress.cu dietgpu/float/GpuFloatInfo.cu)
pids=()
for s in "${SRCS[@]}"; do
  o="$OUT/obj/$(basename "${s%.cu}").o"
  if [ ! -f "$o" ] || [ "$REF/$s" -nt "$o" ]; then
    "$NVCC" "${FLAGS[@]}" -c "$REF/$s" -o "$o" &
    pids+=($!)
  fi
done
for s in dietgpu/utils/DeviceUtils.cpp dietgpu/utils/StackDeviceMemory.cpp; do
  o="$OUT/obj/$(basename "${s%.cpp}").o"
  if [ ! -f "$o" ]; then
    "$NVCC" "${FLAGS[@]}" -x cu -c "$REF/$s" -o "$o" &
    pids+=($!)
  fi
done
"$NVCC" "${FLAGS[@]}" -c "$HERE/ref_harness.cu" -o "$OUT/obj/ref_harness.o" &
pids+=($!)
for p in "${pids[@]}"; do wait "$p"; done
"$NVCC" -shared -o "$OUT/libdietgpu_ref.so" "$OUT"/obj/*.o -lcudart -ccbin /usr/bin/g++
echo "built $OUT/libdietgpu_ref.so"
