// Library-level entry points of libkpf_b200.so.
#include "common.cuh"

extern "C" int kpf_abi_version(void) { return 4; }
