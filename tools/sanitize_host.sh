#!/bin/bash
# usage: bash tools/sanitize_host.sh — the host-side test helpers (fastx_dump: host reader + whole-member
# inflate; inflate_core_test: the device's gzip decoder compiled for the host; member_core_test: one member,
# or with its fourth argument several, decoded in pieces and relayed wave by wave as the device does it, in
# one wave or as many as its fifth argument asks) rebuilt with -fsanitize=address,undefined, their test
# files run against them, the ordinary builds put back.
# Needs a g++ that ships libasan (CXX_SAN, default /usr/bin/g++).
set -e
cd "$(dirname "$0")/.."
CXX_SAN=${CXX_SAN:-/usr/bin/g++}
LIB=sgcount_b200/lib
SAN="-O1 -g -std=c++17 -pthread -fsanitize=address,undefined -fno-omit-frame-pointer"
mkdir -p /tmp/sgc_san && cp $LIB/fastx_dump $LIB/inflate_core_test $LIB/member_core_test /tmp/sgc_san/
trap 'cp /tmp/sgc_san/fastx_dump /tmp/sgc_san/inflate_core_test /tmp/sgc_san/member_core_test '$LIB'/' EXIT
(cd sgcount_b200/host && $CXX_SAN $SAN -o ../lib/fastx_dump fastx_dump.cpp fastx.cpp inflate.cpp -lz &&
  $CXX_SAN $SAN -o ../lib/inflate_core_test inflate_core_test.cpp &&
  $CXX_SAN $SAN -o ../lib/member_core_test member_core_test.cpp)
ASAN_OPTIONS=detect_leaks=0 UBSAN_OPTIONS=print_stacktrace=1:halt_on_error=1 \
  python -m pytest tests/test_host_reader.py tests/test_host_inflate.py tests/test_device_inflate_core.py tests/test_member_inflate_core.py \
  tests/test_multi_member_inflate_core.py tests/test_member_waves_core.py -x -q
