#!/bin/sh
# Host-side code of the product under AddressSanitizer + UndefinedBehaviorSanitizer (no device needed): builds sanitizer variants of libsgs_cuda.so (host halves of
# every .cu: the C ABI, the file readers, the planners) and of the host-logic check library (quadtree_core.h, shared with the kernel) under /tmp/sgs_asan, then runs
# the host-only tests and the reader fuzzers against them.  Any sanitizer report is printed; the script exits non-zero when a test fails.
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
OUT=/tmp/sgs_asan; mkdir -p $OUT/obj
cd $ROOT/sg-slam_b200/csrc
SAN="-fsanitize=address,-fsanitize=undefined,-fno-omit-frame-pointer"
for f in *.cu orb_plan.cpp; do
  b=${f%.*}
  echo "nvcc -O1 -g -std=c++17 -gencode arch=compute_100a,code=sm_100a -Xcompiler -fPIC,-fvisibility=hidden,$SAN --expt-relaxed-constexpr -fmad=false -c -o $OUT/obj/$b.o $f 2>$OUT/obj/$b.log"
done | xargs -P "$(nproc)" -I{} sh -c "{}"
nvcc -gencode arch=compute_100a,code=sm_100a -shared -o $OUT/libsgs_cuda.so $OUT/obj/*.o -cudart static -Xcompiler -fsanitize=address,-fsanitize=undefined
cat > $OUT/run.py <<'PY'
import sys
R = sys.argv[1]
for p in ('tests', 'sg-slam_b200', 'oracle', ''):
    sys.path.insert(0, R + '/' + p)
from pysgs import binding as B
B.LIB_PATH = '/tmp/sgs_asan/libsgs_cuda.so'
import pytest
t = R + '/tests/'
sys.exit(pytest.main(['-q', '-x', '-p', 'no:cacheprovider', t + 'test_fuzz_readers.py', t + 'test_vocabulary_files.py', t + 'test_settings.py', t + 'test_abi_symbols.py', t + 'test_host_wrappers.py', t + 'test_detector.py',
                      '-k', 'not batched_cpu and not product_never']))
PY
export LD_PRELOAD="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)" ASAN_OPTIONS=detect_leaks=0 UBSAN_OPTIONS=print_stacktrace=1
python $OUT/run.py $ROOT
