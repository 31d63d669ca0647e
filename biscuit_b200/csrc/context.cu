// Context lifecycle of libbiscuit_b200 (one bq_ctx per GPU / host thread).
#include "encoded.cuh"

static thread_local std::string g_create_error;

extern "C" {

int bq_abi_version(void) { return BQ_ABI_VERSION; }

int bq_create(int device, bq_ctx** out) {
  if (!out) return BQ_ERR_ARG;
  *out = nullptr;
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count == 0) {
    g_create_error = std::string("no CUDA device available: ") + cudaGetErrorString(e);
    cudaGetLastError();
    return BQ_ERR_CUDA;
  }
  if (device < 0 || device >= count) {
    g_create_error = "device index out of range";
    return BQ_ERR_ARG;
  }
  if ((e = cudaSetDevice(device)) != cudaSuccess) {
    g_create_error = std::string("cudaSetDevice: ") + cudaGetErrorString(e);
    return BQ_ERR_CUDA;
  }
  cudaDeviceProp prop;
  if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_create_error = std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e);
    return BQ_ERR_CUDA;
  }
  if (prop.major != 10) {
    char buf[256];
    snprintf(buf, sizeof(buf), "libbiscuit_b200 is built for sm_100a only; device %d is sm_%d%d (%s)", device,
             prop.major, prop.minor, prop.name);
    g_create_error = buf;
    return BQ_ERR_CUDA;
  }
  bq_ctx* ctx = new bq_ctx();
  ctx->device = device;
  ctx->num_sms = prop.multiProcessorCount;
  if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_create_error = std::string("cudaStreamCreate: ") + cudaGetErrorString(e);
    delete ctx;
    return BQ_ERR_CUDA;
  }
  // keep memory freed by cudaFreeAsync cached in the default pool (per-call thresholding temporaries are re-allocated
  // on every apply / detect; trimming the pool at each synchronisation would turn them back into cudaMalloc calls)
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    uint64_t keep = UINT64_MAX;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
  cudaGetLastError();
  *out = ctx;
  return BQ_OK;
}

void bq_destroy(bq_ctx* ctx) {
  if (!ctx) return;
  bq_comm_destroy(ctx);                     // no-op without a communicator
  cudaSetDevice(ctx->device);
  if (ctx->stream) {
    cudaStreamSynchronize(ctx->stream);
    cudaStreamDestroy(ctx->stream);
  }
  if (ctx->scratch) cudaFree(ctx->scratch);
  delete ctx->jpeg;
  delete ctx->png;
  if (ctx->pinned) cudaFreeHost(ctx->pinned);
  delete ctx;
}

const char* bq_last_error(bq_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int64_t bq_launch_count(bq_ctx* ctx) { return ctx ? ctx->launches : 0; }

int bq_sync(bq_ctx* ctx) {
  if (!ctx) return BQ_ERR_ARG;
  BQ_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
  return BQ_OK;
}

void* bq_stream(bq_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }

}  // extern "C"
