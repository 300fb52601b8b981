#!/bin/bash
# Build the library under another name with extra -D flags: kernel A/B runs without touching the in-tree libevgsim.so.
#   tools/build_variant.sh NAME [-DEVG_CHECKED ...]   ->  build/libevgsim_NAME.so
# Select it with EVGSIM_LIB=build/libevgsim_NAME.so (see tools/ab_variants.sh).  The sources and nvcc flags are those of
# __graft_entry__.build().
set -e
cd "$(dirname "$0")/.."
name=$1; shift
mkdir -p build
python3 -c 'import sys, __graft_entry__ as g; g.compile_library(sys.argv[1], sys.argv[2:], force=True)' "build/libevgsim_$name.so" "$@"
echo built build/libevgsim_$name.so
