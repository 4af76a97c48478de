#!/bin/bash
# The kernels' sources (pass 1, pass 2, single-stream route, containers, chunked input, compression,
# and the block-level kernels of tests/cpu_emu/emu_block.cpp) compiled for the host under
# AddressSanitizer + UBSan and run through the emulation tests: every golden family, truncation /
# bit-flip / capacity sweep included.  CPU only.
set -e
cd "$(dirname "$0")/.."
LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0 SFB_EMU_ASAN=1 \
  python -m pytest tests/test_kernel_logic_cpu.py tests/test_block_kernels_cpu.py -x -q "$@"
rm -f tests/cpu_emu/*_asan.so
