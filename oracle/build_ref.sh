#!/usr/bin/env bash
# Builds the REFERENCE's own CUDA kernels (lib/ops/raymarching, lib/ops/shencoder) from the sources where they lie under
# /root/reference into oracle/_ref/ (git-ignored, travels to the GPU box), with ONE flag change: -std=c++14 -> -std=c++17
# (PyTorch 2.11 headers need C++17; SURVEY.md F6).  Used by tests/golden/make_golden_ref_kernels.py to store the outputs
# tests/test_ref_gpu.py compares against, and by tests/perf/ref_gpu_baseline.py as the reference-GPU baseline.
# No reference source is copied into the repo.
set -euo pipefail
REF=${REF:-/root/reference}
HERE="$(cd "$(dirname "$0")" && pwd)"
OUT="$HERE/_ref"
mkdir -p "$OUT"
PY=${PYTHON:-python}
TORCH_INC=$($PY -c "import torch.utils.cpp_extension as c; print(' '.join('-I'+p for p in c.include_paths()))")
PY_INC=$($PY -c "import sysconfig; print('-I'+sysconfig.get_paths()['include'])")
TORCH_LIB=$($PY -c "import torch, os; print(os.path.join(os.path.dirname(torch.__file__), 'lib'))")
EXT=$($PY -c "import sysconfig; print(sysconfig.get_config_var('EXT_SUFFIX'))")
COMMON="-O3 -std=c++17 -U__CUDA_NO_HALF_OPERATORS__ -U__CUDA_NO_HALF_CONVERSIONS__ -U__CUDA_NO_HALF2_OPERATORS__ --expt-relaxed-constexpr \
 -gencode arch=compute_100a,code=sm_100a $TORCH_INC $PY_INC -Xcompiler -fPIC -D_GLIBCXX_USE_CXX11_ABI=1"
build_one () {   # name srcdir module
  local name=$1 dir=$2 mod=$3
  nvcc $COMMON -DTORCH_EXTENSION_NAME=$mod -c "$dir/src/$name.cu" -o "$OUT/$name.o"
  g++ -O3 -std=c++17 -fPIC $TORCH_INC $PY_INC -DTORCH_EXTENSION_NAME=$mod -D_GLIBCXX_USE_CXX11_ABI=1 -c "$dir/src/bindings.cpp" -o "$OUT/${name}_bind.o"
  g++ -shared "$OUT/$name.o" "$OUT/${name}_bind.o" -L"$TORCH_LIB" -ltorch -ltorch_cpu -ltorch_cuda -lc10 -lc10_cuda -ltorch_python \
      -L/usr/local/cuda/lib64 -lcudart -Wl,-rpath,"$TORCH_LIB" -o "$OUT/$mod$EXT"
  rm -f "$OUT/$name.o" "$OUT/${name}_bind.o"
}
build_one raymarching "$REF/lib/ops/raymarching" _raymarching
build_one shencoder "$REF/lib/ops/shencoder" _shencoder
ls -la "$OUT"
