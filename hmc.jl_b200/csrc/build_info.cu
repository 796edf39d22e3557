// build_info.cu — the identity of this build: ABI version and the hash of every source file the library was compiled from
// (hmc.jl_b200/build.py::source_hash passes it as HMC_SRC_HASH).  Hosts compare it with the sources next to them, so a stale
// libhmcgpu.so can never be measured or tested by mistake.
#include "../../include/hmcgpu.h"
#ifndef HMC_SRC_HASH
#define HMC_SRC_HASH "unknown"
#endif
extern "C" int hmcgpu_version(void) { return 600; }
extern "C" const char* hmcgpu_build_info(void) { return "600;" HMC_SRC_HASH; }
