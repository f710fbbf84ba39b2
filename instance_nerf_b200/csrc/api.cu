// Version / error-string entry points of libinerf_b200.
#include "common.cuh"

extern "C" int inerf_version(void) { return 1001; }

extern "C" const char* inerf_error_string(int code) {
    if (code > 0) return cudaGetErrorString((cudaError_t)code);
    switch (code) {
        case INERF_OK: return "ok";
        case INERF_ERR_NULL: return "inerf: required pointer is NULL";
        case INERF_ERR_SIZE: return "inerf: size or count out of range";
        case INERF_ERR_UNSUPPORTED: return "inerf: unsupported configuration";
        case INERF_ERR_WORKSPACE: return "inerf: workspace too small";
        case INERF_ERR_ALIGN: return "inerf: pointer not sufficiently aligned";
        default: return "inerf: unknown error";
    }
}
