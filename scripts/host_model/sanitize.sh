#!/bin/bash
# Two CPU builds under ASan + UBSan, driven by the tests:
# - the host build of the product's device headers (tests/host_device), driven by tests/test_device_source_on_host.py:
#   closest-hit queries, BVH traversals (stack of RBRT_STACK entries, leaf decoding, 16-bit node decode), scatter, complete renders;
# - the CPU oracle (oracle/rbrt_oracle.cpp), driven by the same module and by the renders of paths longer than 64 bounces, up to
#   max_depth 1024 (tests/test_oracle_quirks.py, tests/test_oracle_numpy_crosscheck.py).  A stack overwrite in the oracle is silent
#   in a plain build; this is where it shows.
# compute-sanitizer is closed on the GPU pool; this is the memory-safety evidence available for that code.
set -e
cd "$(dirname "$0")/../.."
hd=tests/host_device
mkdir -p $hd/build oracle/build
SAN="-fsanitize=address,undefined -fno-sanitize-recover=undefined"
g++ -O1 -g -std=c++17 -ffp-contract=off -fno-fast-math -mno-fma -DRBRT_LDG128 $SAN \
    -Wno-unknown-pragmas -fPIC -shared -I $hd -I rbrt_b200/csrc -o $hd/build/libhost_device.so $hd/harness.cpp
touch $hd/build/libhost_device.so
g++ -O1 -g -mavx -ffp-contract=off -fno-fast-math -std=c++17 -fPIC -Wall -Wno-unused-function -pthread $SAN \
    -shared -o oracle/build/librbrt_oracle.so oracle/rbrt_oracle.cpp
LD_PRELOAD="$(gcc -print-file-name=libasan.so) $(gcc -print-file-name=libubsan.so)" ASAN_OPTIONS=detect_leaks=0 \
    python -m pytest tests/test_device_source_on_host.py tests/test_oracle_quirks.py tests/test_oracle_numpy_crosscheck.py -x -q --capture=sys || rc=$?   # sys: a sanitizer report on fd 2 reaches the terminal
rm -f $hd/build/libhost_device.so                     # the next test run rebuilds the plain library
rm -f oracle/build/librbrt_oracle.so && make -s -C oracle
exit ${rc:-0}
