// Context, error reporting.
#include "common.cuh"
#include <stdarg.h>
#include <stdlib.h>

static thread_local char g_err[1024] = "";

void sg_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" {

int sg_version(void) { return 100; }

const char* sg_last_error(void) { return g_err; }

int sg_ctx_create(int device, void* cuda_stream, sg_ctx** out) {
  SG_REQUIRE(out != nullptr, "sg_ctx_create: out is NULL");
  int count = 0;
  SG_CHECK_CUDA(cudaGetDeviceCount(&count));
  SG_REQUIRE(device >= 0 && device < count, "sg_ctx_create: device %d out of range (%d devices)", device, count);
  SG_CHECK_CUDA(cudaSetDevice(device));
  cudaDeviceProp prop;
  SG_CHECK_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    sg_set_error("sg_ctx_create: device %d is sm_%d%d; libsgan is built for sm_100a only", device, prop.major,
                 prop.minor);
    return SG_ERR_UNSUPPORTED;
  }
  sg_ctx* c = (sg_ctx*)calloc(1, sizeof(sg_ctx));
  c->device = device;
  c->stream = (cudaStream_t)cuda_stream;
  c->num_sms = prop.multiProcessorCount;
  c->encode_tiled = nullptr;
  c->launches = 0;
  c->conv_split_tail = 1;
  // the ONE device allocation libsgan makes: the fixed workspace of the deterministic reductions (common.cuh)
  cudaError_t e1 = cudaMalloc((void**)&c->det_scratch, SG_DET_SCRATCH_BYTES);
  cudaError_t e2 = e1 == cudaSuccess ? cudaMalloc((void**)&c->det_tickets, SG_DET_TICKETS * sizeof(unsigned int)) : e1;
  cudaError_t e3 = e2 == cudaSuccess ? cudaMemset(c->det_tickets, 0, SG_DET_TICKETS * sizeof(unsigned int)) : e2;
  if (e3 != cudaSuccess) {
    sg_set_error("sg_ctx_create: workspace allocation failed: %s", cudaGetErrorString(e3));
    if (c->det_scratch) cudaFree(c->det_scratch);
    if (c->det_tickets) cudaFree(c->det_tickets);
    free(c);
    return SG_ERR_CUDA;
  }
  *out = c;
  return SG_OK;
}

int sg_ctx_destroy(sg_ctx* ctx) {
  if (ctx) {
    for (int i = 0; i < ctx->n_aux; ++i) {
      cudaStreamDestroy(ctx->aux_stream[i]);
      cudaEventDestroy(ctx->aux_join[i]);
    }
    if (ctx->n_aux) cudaEventDestroy(ctx->aux_fork);
    if (ctx->det_scratch) cudaFree(ctx->det_scratch);
    if (ctx->det_tickets) cudaFree(ctx->det_tickets);
    free(ctx);
  }
  return SG_OK;
}

int sg_ctx_set_stream(sg_ctx* ctx, void* cuda_stream) {
  SG_REQUIRE(ctx != nullptr, "ctx is NULL");
  ctx->stream = (cudaStream_t)cuda_stream;
  return SG_OK;
}

int sg_ctx_sync(sg_ctx* ctx) {
  SG_REQUIRE(ctx != nullptr, "ctx is NULL");
  SG_CHECK_CUDA(cudaStreamSynchronize(ctx->stream));
  return SG_OK;
}

long long sg_ctx_launch_count(sg_ctx* ctx) { return ctx ? ctx->launches : -1; }

/* zero `bytes` of device memory on the context's stream (a memset node, no kernel): gradient buckets at the start of a step */
int sg_zero(sg_ctx* ctx, void* ptr, size_t bytes) {
  SG_REQUIRE(ctx != nullptr && (ptr != nullptr || bytes == 0), "sg_zero: bad args");
  if (bytes) SG_CHECK_CUDA(cudaMemsetAsync(ptr, 0, bytes, ctx->stream));
  return SG_OK;
}

int sg_ctx_set_speed_mode(sg_ctx* ctx, int on) {
  SG_REQUIRE(ctx != nullptr, "ctx is NULL");
  ctx->speed_mode = on ? 1 : 0;
  return SG_OK;
}

int sg_ctx_set_conv_split_tail(sg_ctx* ctx, int on) {
  SG_REQUIRE(ctx != nullptr, "ctx is NULL");
  ctx->conv_split_tail = on ? 1 : 0;
  return SG_OK;
}

}  // extern "C"

// layout guard for the ctypes mirror of sg_conv_desc
extern "C" int sg_sizeof_conv_desc(void) { return (int)sizeof(sg_conv_desc); }

// ---------------------------------------------------------------------------------------------------
// CRC32C (Castagnoli), slicing-by-8, host side: TensorFlow checkpoints protect every tensor and every index block with it
// (tf_checkpoint.py reads / writes the reference's save_weights files: data_utils.py:346-348)
// ---------------------------------------------------------------------------------------------------
static uint32_t g_crc_tab[8][256];
static bool g_crc_init = false;
static void crc_init() {
  for (uint32_t i = 0; i < 256; ++i) {
    uint32_t c = i;
    for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1) ? 0x82F63B78u : 0u);
    g_crc_tab[0][i] = c;
  }
  for (uint32_t i = 0; i < 256; ++i)
    for (int t = 1; t < 8; ++t) g_crc_tab[t][i] = (g_crc_tab[t - 1][i] >> 8) ^ g_crc_tab[0][g_crc_tab[t - 1][i] & 0xFF];
  g_crc_init = true;
}

extern "C" unsigned int sg_crc32c(const void* data, size_t n, unsigned int crc) {
  if (!g_crc_init) crc_init();
  const unsigned char* p = (const unsigned char*)data;
  uint32_t c = crc ^ 0xFFFFFFFFu;
  while (n && ((uintptr_t)p & 7)) { c = g_crc_tab[0][(c ^ *p++) & 0xFF] ^ (c >> 8); --n; }
  while (n >= 8) {
    uint64_t v;
    memcpy(&v, p, 8);
    uint32_t lo = (uint32_t)v ^ c, hi = (uint32_t)(v >> 32);
    c = g_crc_tab[7][lo & 0xFF] ^ g_crc_tab[6][(lo >> 8) & 0xFF] ^ g_crc_tab[5][(lo >> 16) & 0xFF] ^ g_crc_tab[4][lo >> 24] ^
        g_crc_tab[3][hi & 0xFF] ^ g_crc_tab[2][(hi >> 8) & 0xFF] ^ g_crc_tab[1][(hi >> 16) & 0xFF] ^ g_crc_tab[0][hi >> 24];
    p += 8;
    n -= 8;
  }
  while (n--) c = g_crc_tab[0][(c ^ *p++) & 0xFF] ^ (c >> 8);
  return c ^ 0xFFFFFFFFu;
}
