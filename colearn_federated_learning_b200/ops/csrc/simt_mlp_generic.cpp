// mlp_generic.cu compiled for the CPU through host_shim.h (thread-block clusters emulated) — see simt_emul.cpp
#define COLEARN_HOST_SHIM 1
#include "host_shim.h"

#include "mlp_generic.cu"   // NOLINT(bugprone-suspicious-include): the kernel source itself
