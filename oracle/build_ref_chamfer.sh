#!/usr/bin/env bash
# TEST INFRASTRUCTURE — not product code.
#
# Compiles the UNMODIFIED reference Chamfer extension
# ($NVSF_REFERENCE/nvsf/nerf/chamfer3D/{chamfer3D.cu,chamfer_cuda.cpp}, NVSF_REFERENCE = a checkout
# of the reference project) for sm_100a into oracle/_ref/chamfer_3D_ref.so, from the sources where
# they lie (nothing is copied).  The reference JIT-builds these two files with
# torch.utils.cpp_extension.load (dist_chamfer_3D.py:27-35); this is the same compile with an
# explicit -gencode for B200.  Without the reference sources the script is a no-op and a prebuilt
# .so, if any, is used by oracle/make_golden_chamfer.py and the -m gpu tests.
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
SRC=${NVSF_REFERENCE:-}/nvsf/nerf/chamfer3D
OUT="$HERE/_ref"
if [ ! -d "$SRC" ]; then
    echo "[build_ref_chamfer] $SRC not present (GPU box?) - skipping"; exit 0
fi
mkdir -p "$OUT"
if [ -f "$OUT/chamfer_3D_ref.so" ] && [ "$OUT/chamfer_3D_ref.so" -nt "$SRC/chamfer3D.cu" ] \
   && [ "${1:-}" != "--force" ]; then
    echo "[build_ref_chamfer] up to date"; exit 0
fi
PY=${PYTHON:-python}
TORCH_DIR=$($PY -c 'import torch,os;print(os.path.dirname(torch.__file__))')
PY_INC=$($PY -c 'import sysconfig;print(sysconfig.get_paths()["include"])')
INC="-I$TORCH_DIR/include -I$TORCH_DIR/include/torch/csrc/api/include -I$PY_INC -I/usr/local/cuda/include"
DEFS="-DTORCH_EXTENSION_NAME=chamfer_3D_ref -DTORCH_API_INCLUDE_EXTENSION_H -D_GLIBCXX_USE_CXX11_ABI=1"
nvcc -c "$SRC/chamfer3D.cu" -o "$OUT/chamfer3D_ref.o" -O3 -std=c++17 \
    -gencode arch=compute_100a,code=sm_100a --expt-relaxed-constexpr -Xcompiler -fPIC $INC $DEFS &
g++ -c "$SRC/chamfer_cuda.cpp" -o "$OUT/chamfer_cuda_ref.o" -O3 -std=c++17 -fPIC $INC $DEFS &
wait
g++ -shared "$OUT/chamfer3D_ref.o" "$OUT/chamfer_cuda_ref.o" -o "$OUT/chamfer_3D_ref.so" \
    -L"$TORCH_DIR/lib" -L/usr/local/cuda/lib64 \
    -lc10 -ltorch -ltorch_cpu -ltorch_python -lc10_cuda -ltorch_cuda -lcudart \
    -Wl,-rpath,"$TORCH_DIR/lib"
rm -f "$OUT/chamfer3D_ref.o" "$OUT/chamfer_cuda_ref.o"
echo "[build_ref_chamfer] built $OUT/chamfer_3D_ref.so"
