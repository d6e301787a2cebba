#!/usr/bin/env bash
# TEST INFRASTRUCTURE — not product code.
#
# Compiles the UNMODIFIED reference ray-marching extension
# ($NVSF_REFERENCE/nvsf/nerf/raymarching/src/{raymarching.cu,bindings.cpp}, NVSF_REFERENCE = a
# checkout of the reference project) for sm_100a into oracle/_ref/_raymarching_ref.so.  Sources
# are compiled where they lie; nothing is copied into this repository.  The flags are the
# reference's own setup.py flags (nvsf/nerf/raymarching/setup.py:7-13) plus an
# explicit -gencode for B200.  The result is a torch/pybind extension that can
# only EXECUTE on a GPU; `-m gpu` tests use it as the live oracle when
# present (oracle/_ref/ is git-ignored).
#
# Without the reference sources this script is a no-op and a prebuilt .so, if any, is used.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
SRC=${NVSF_REFERENCE:-}/nvsf/nerf/raymarching/src
OUT="$HERE/_ref"
if [ ! -d "$SRC" ]; then
    echo "[build_ref] $SRC not present (GPU box?) - skipping"; exit 0
fi
mkdir -p "$OUT"
if [ -f "$OUT/_raymarching_ref.so" ] && [ "$OUT/_raymarching_ref.so" -nt "$SRC/raymarching.cu" ] \
   && [ "${1:-}" != "--force" ]; then
    echo "[build_ref] up to date"; exit 0
fi
PY=${PYTHON:-python}
TORCH_DIR=$($PY -c 'import torch,os;print(os.path.dirname(torch.__file__))')
PY_INC=$($PY -c 'import sysconfig;print(sysconfig.get_paths()["include"])')
EXT_SUFFIX=.so
INC="-I$TORCH_DIR/include -I$TORCH_DIR/include/torch/csrc/api/include -I$PY_INC -I/usr/local/cuda/include"
DEFS="-DTORCH_EXTENSION_NAME=_raymarching_ref -DTORCH_API_INCLUDE_EXTENSION_H -D_GLIBCXX_USE_CXX11_ABI=1"
nvcc -c "$SRC/raymarching.cu" -o "$OUT/raymarching_ref.o" -O3 -std=c++17 \
    -U__CUDA_NO_HALF_OPERATORS__ -U__CUDA_NO_HALF_CONVERSIONS__ -U__CUDA_NO_HALF2_OPERATORS__ \
    -gencode arch=compute_100a,code=sm_100a --expt-relaxed-constexpr \
    -Xcompiler -fPIC $INC $DEFS &
g++ -c "$SRC/bindings.cpp" -o "$OUT/bindings_ref.o" -O3 -std=c++17 -fPIC $INC $DEFS &
wait
g++ -shared "$OUT/raymarching_ref.o" "$OUT/bindings_ref.o" -o "$OUT/_raymarching_ref.so" \
    -L"$TORCH_DIR/lib" -L/usr/local/cuda/lib64 \
    -lc10 -ltorch -ltorch_cpu -ltorch_python -lc10_cuda -ltorch_cuda -lcudart \
    -Wl,-rpath,"$TORCH_DIR/lib"
rm -f "$OUT/raymarching_ref.o" "$OUT/bindings_ref.o"
echo "[build_ref] built $OUT/_raymarching_ref.so"
