// Library-level entry points of libjt_vm.so.
#include "jt_common.cuh"
#include "../../include/jt_vm.h"

namespace jt { long long g_launches = 0; }

extern "C" const char* jt_strerror(int code) {
    switch (code) {
        case JT_OK: return "ok";
        case JT_ERR_ARG: return "invalid argument (null pointer, bad size or alignment)";
        case JT_ERR_LAUNCH: return "CUDA kernel launch failed";
        case JT_ERR_UNSUPPORTED: return "configuration not supported by this kernel";
        default: return "unknown error";
    }
}
extern "C" int jt_version(void) { return 4; }
extern "C" long long jt_launch_count(void) { return jt::g_launches; }
