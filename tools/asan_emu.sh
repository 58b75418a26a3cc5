#!/bin/bash
# the kernel-logic build (tests/emu) under AddressSanitizer: every kernel body, the ABI and the fetches with heap checking
set -e
cd "$(dirname "$0")/.."
g++ -O1 -g -std=c++17 -fPIC -shared -DAGPU_EMU -x c++ -w -pthread -fsanitize=address -fno-omit-frame-pointer -Iinclude \
	-o /tmp/libaletsch_emu_asan.so aletsch_b200/csrc/aletsch_gpu.cu
LD_PRELOAD=$(g++ -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0 ALETSCH_EMU_LIB=/tmp/libaletsch_emu_asan.so \
	python -m pytest tests/test_emu_parity.py tests/test_fuzz.py tests/test_adapter_transcripts.py tests/test_pipeline.py tests/test_cluster_pass.py tests/test_cli.py tests/test_group_phase_set.py tests/test_param_sweep.py -x -q -m "not gpu" "$@"
