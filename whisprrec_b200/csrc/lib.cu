// Library bookkeeping: version, error strings, the device workspace.
#include "common.cuh"

extern "C" int wr_version(void) { return WR_VERSION; }

extern "C" const char *wr_error_string(int code) {
    switch (code) {
        case WR_OK: return "ok";
        case WR_E_NULL: return "a required pointer is NULL";
        case WR_E_SIZE: return "negative or inconsistent size";
        case WR_E_DIM: return "unsupported embedding size (needs D % 4 == 0; eval needs D in {16,32,64,128,256})";
        case WR_E_TOPK: return "k outside [1, 32]";
        case WR_E_ALIGN: return "table pointer not 16-byte aligned";
        case WR_E_PRECISION: return "unknown or unavailable scoring precision";
        default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown whisprrec_b200 error";
    }
}

extern "C" size_t wr_workspace_bytes(void) { return sizeof(WrWorkspace); }

extern "C" int wr_workspace_init(void *ws, void *stream) {
    if (!ws) return WR_E_NULL;
    return (int)cudaMemsetAsync(ws, 0, sizeof(WrWorkspace), (cudaStream_t)stream);
}

extern "C" int wr_status(void *ws, uint32_t *host_status, void *stream) {
    if (!ws || !host_status) return WR_E_NULL;
    cudaStream_t st = (cudaStream_t)stream;
    cudaError_t e = cudaMemcpyAsync(host_status, ws, sizeof(uint32_t), cudaMemcpyDeviceToHost, st);
    if (e != cudaSuccess) return (int)e;
    e = cudaMemsetAsync(ws, 0, sizeof(uint32_t), st);
    if (e != cudaSuccess) return (int)e;
    return (int)cudaStreamSynchronize(st);
}
