#!/bin/bash
# Builds the library under AddressSanitizer + UBSan (host code; the device code is compiled but never
# launched), dumps the golden fixtures as seed files and runs tests/native/host_parse_fuzz.cpp.  CPU only.
set -e
ROOT=$(cd "$(dirname "$0")/../.." && pwd)
HERE=$ROOT/lilliput_b200/csrc
OUT=${LP_ASAN_DIR:-/tmp/asan}
ITERS=${1:-200000}
mkdir -p $OUT/build $OUT/seeds
SAN=-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer,-fno-sanitize-recover=undefined
FLAGS="-gencode arch=compute_100a,code=sm_100a -O1 -g -std=c++17 -Xcompiler -fPIC,$SAN -I$ROOT/include -I$ROOT/lilliput_b200/host -I$HERE"
cd $OUT/build
for f in resize jpeg_decode jpeg_huff_parallel jpeg_encode png_decode png_encode gif_decode webp_decode webp_encode pixel_ops abi_opencv batch; do
  [ $f.o -nt $HERE/$f.cu ] || ( nvcc $FLAGS -c $HERE/$f.cu -o $f.o ) &
done
[ jpeg_parse.o -nt $HERE/jpeg_parse.cpp ] || ( nvcc $FLAGS -x cu -c $HERE/jpeg_parse.cpp -o jpeg_parse.o ) &
[ png_parse.o -nt $HERE/png_parse.cpp ] || ( nvcc $FLAGS -x cu -c $HERE/png_parse.cpp -o png_parse.o ) &
[ lilliput_host.o -nt $ROOT/lilliput_b200/host/lilliput_host.cpp ] || ( nvcc $FLAGS -x cu -c $ROOT/lilliput_b200/host/lilliput_host.cpp -o lilliput_host.o ) &
wait
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $OUT/liblp_asan.so *.o -cudart static -Xcompiler $SAN -Xlinker -Bsymbolic
g++ -O1 -g -std=c++17 -fsanitize=address,undefined -fno-omit-frame-pointer -I$ROOT/include -I$HERE \
    -I${CUDA_HOME:-/usr/local/cuda}/include \
    $ROOT/tests/native/host_parse_fuzz.cpp -o $OUT/host_parse_fuzz -L$OUT -llp_asan -Wl,-rpath,$OUT
python - <<PY
import numpy as np, os, sys
root, out = "$ROOT", "$OUT/seeds"
sys.path.insert(0, root)
from tests.golden import load  # merges the parts of a set stored as <name>.npz, <name>_2.npz, ...
n = 0
for f, prefixes in [("golden", ("gif_", "png_", "jpeg_", "jpegvar_", "c1_input", "c6_input")),
                    ("webp_golden", ("webp_",)), ("jpeg_multiscan_golden", ("jpg_",)),
                    ("png_adam7_golden", ("png_",)), ("jpeg_optimized_golden", ("jpg_",)),
                    ("gif_encode_golden", ("out_",))]:
    g = load(f)
    for k in g.files:
        a = g[k]
        if k.startswith(prefixes) and a.dtype == np.uint8 and a.ndim == 1 and 16 <= a.size <= 60000:
            open(os.path.join(out, f"{n:04d}_{k}"), "wb").write(a.tobytes())
            n += 1
print(n, "seed files")
PY
ASAN_OPTIONS=detect_leaks=1:allocator_may_return_null=1:max_allocation_size_mb=4096 $OUT/host_parse_fuzz $ITERS $OUT/seeds/*
