#!/usr/bin/env bash
# TEST INFRASTRUCTURE.  Builds the reference's OWN torch extensions — `r3dg_rasterization._C`
# (r3dg-rasterization/setup.py:21-33: rasterizer_impl.cu forward.cu backward.cu rasterize_points.cu
# ext.cpp) and `bvh_tracing._C` (bvh/setup.py:12-26: bvh.cu trace.cu construct.cu bindings.cpp) —
# for sm_100 with the reference's flags, from the sources where they lie under /root/reference, into
# oracle/_ref/ext/ (git-ignored; travels to the GPU box with gpurun), and drops the reference's two
# Python wrapper files (+ the two utils modules they import) into oracle/_ref/py/.
#
# With these, `bench.py --impl reference` and tests/test_dropin_gpu.py run the STOCK code path:
# the reference's Python wrapper -> its pybind module -> its torch glue -> its kernels.  Nothing
# here is product code, and nothing is copied into git history.  ~15 min of nvcc (torch headers).
set -euo pipefail
HERE="$(cd "$(dirname "${BASH_SOURCE[0]}")" && pwd)"
REF="${R3DG_REFERENCE:-/root/reference}"
OUT="$HERE/_ref"
[ -d "$REF" ] || { echo "[build_ref_ext] $REF absent — skipping (prebuilt oracle/_ref/ext is used if present)"; exit 0; }
PY="${PYTHON:-python}"
NVCC="${NVCC:-/usr/local/cuda/bin/nvcc}"
mkdir -p "$OUT/ext/r3dg_rasterization" "$OUT/ext/bvh_tracing" "$OUT/py/gaussian_renderer" "$OUT/py/bvh" "$OUT/py/utils" "$OUT/obj"

# the wrapper sources (git-ignored copies; loaded by file path in the tests / reference arm)
cp "$REF/gaussian_renderer/r3dg_rasterization.py" "$OUT/py/gaussian_renderer/r3dg_rasterization.py"
cp "$REF/bvh/__init__.py" "$OUT/py/bvh/__init__.py"
cp "$REF/utils/system_utils.py" "$REF/utils/general_utils.py" "$REF/utils/sh_utils.py" "$REF/utils/graphics_utils.py" "$OUT/py/utils/"
touch "$OUT/py/utils/__init__.py"
: > "$OUT/ext/r3dg_rasterization/__init__.py"
: > "$OUT/ext/bvh_tracing/__init__.py"

TORCH_INC=$($PY - <<'EOF'
import warnings; warnings.filterwarnings("ignore")
import sysconfig, torch.utils.cpp_extension as c
print(" ".join("-I" + p for p in c.include_paths("cuda")) + " -I" + sysconfig.get_paths()["include"])
EOF
)
TORCH_LIB=$($PY -c "import os, torch; print(os.path.join(os.path.dirname(torch.__file__), 'lib'))" 2>/dev/null)
ARCH="-gencode arch=compute_100,code=sm_100"
# what torch's BuildExtension adds to every nvcc line
TORCHISH="-D__CUDA_NO_HALF_OPERATORS__ -D__CUDA_NO_HALF_CONVERSIONS__ -D__CUDA_NO_BFLOAT16_CONVERSIONS__ -D__CUDA_NO_HALF2_OPERATORS__ --expt-relaxed-constexpr -std=c++17 -DTORCH_API_INCLUDE_EXTENSION_H -D_GLIBCXX_USE_CXX11_ABI=1"
RAS="$REF/r3dg-rasterization"
BVH="$REF/bvh"

if [ ! -f "$OUT/ext/r3dg_rasterization/_C.so" ]; then
  echo "[build_ref_ext] r3dg_rasterization._C"
  for f in cuda_rasterizer/rasterizer_impl cuda_rasterizer/forward cuda_rasterizer/backward rasterize_points; do
    o="$OUT/obj/ras_$(basename $f).o"
    $NVCC $ARCH -O3 $TORCHISH -DTORCH_EXTENSION_NAME=_C --pre-include cstdint -I"$RAS/third_party/glm" -I"$RAS" $TORCH_INC \
        -Xcompiler -fPIC -c "$RAS/$f.cu" -o "$o" &
  done
  g++ -O3 -std=c++17 -fPIC -DTORCH_EXTENSION_NAME=_C -DTORCH_API_INCLUDE_EXTENSION_H -D_GLIBCXX_USE_CXX11_ABI=1 -I"$RAS" $TORCH_INC \
      -c "$RAS/ext.cpp" -o "$OUT/obj/ras_ext.o" &
  wait
  g++ -shared -o "$OUT/ext/r3dg_rasterization/_C.so" "$OUT"/obj/ras_*.o -L"$TORCH_LIB" -L/usr/local/cuda/lib64 \
      -lc10 -lc10_cuda -ltorch_cpu -ltorch_cuda -ltorch -ltorch_python -lcudart -Wl,-rpath,"$TORCH_LIB"
fi

if [ ! -f "$OUT/ext/bvh_tracing/_C.so" ]; then
  echo "[build_ref_ext] bvh_tracing._C (construct.cu: the one-line '-> aabb_type' patched copy, SURVEY §8c-addendum)"
  sed '166s/rhs)[[:space:]]*{/rhs) -> aabb_type {/' "$BVH/src/construct.cu" > "$OUT/construct_patched.cu"
  diff "$BVH/src/construct.cu" "$OUT/construct_patched.cu" || true
  $NVCC $ARCH -O3 $TORCHISH -DTORCH_EXTENSION_NAME=_C --expt-extended-lambda -I"$BVH/include" $TORCH_INC -Xcompiler -fPIC \
      -c "$BVH/src/bvh.cu" -o "$OUT/obj/bvh_bvh.o" &
  $NVCC $ARCH -O3 $TORCHISH -DTORCH_EXTENSION_NAME=_C --expt-extended-lambda -I"$BVH/include" $TORCH_INC -Xcompiler -fPIC \
      -c "$BVH/src/trace.cu" -o "$OUT/obj/bvh_trace.o" &
  $NVCC $ARCH -O3 $TORCHISH -DTORCH_EXTENSION_NAME=_C --expt-extended-lambda -I"$BVH/include" $TORCH_INC -Xcompiler -fPIC \
      -c "$OUT/construct_patched.cu" -o "$OUT/obj/bvh_construct.o" &
  g++ -O3 -std=c++17 -fPIC -DTORCH_EXTENSION_NAME=_C -DTORCH_API_INCLUDE_EXTENSION_H -D_GLIBCXX_USE_CXX11_ABI=1 -I"$BVH/include" $TORCH_INC \
      -c "$BVH/src/bindings.cpp" -o "$OUT/obj/bvh_bindings.o" &
  wait
  g++ -shared -o "$OUT/ext/bvh_tracing/_C.so" "$OUT"/obj/bvh_*.o -L"$TORCH_LIB" -L/usr/local/cuda/lib64 \
      -lc10 -lc10_cuda -ltorch_cpu -ltorch_cuda -ltorch -ltorch_python -lcudart -Wl,-rpath,"$TORCH_LIB"
fi
rm -rf "$OUT/obj"
echo "[build_ref_ext] done: $(ls "$OUT/ext"/*/)"
