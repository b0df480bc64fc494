// api.cu - version / error string / device query of the C ABI (include/atvs.h).
#include "common.cuh"
#include <stdarg.h>

static thread_local char g_err[512] = "";

void atvs_set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

extern "C" int atvs_version(void) { return 100; }
extern "C" const char* atvs_last_error(void) { return g_err; }
extern "C" int atvs_device_sm_count(void) { return atvs_num_sms(); }

// CRC-32C (Castagnoli), slice-by-8 on the host: the tensor checksums of a TensorFlow V2 checkpoint (ckpt.py) are
// verified for every tensor, not only the small ones a pure-Python loop can afford
static unsigned g_crc_tab[8][256];
static bool g_crc_init = false;
extern "C" unsigned atvs_crc32c(const void* data, size_t n, unsigned crc) {
    if (!g_crc_init) {
        for (unsigned i = 0; i < 256; ++i) {
            unsigned c = i;
            for (int k = 0; k < 8; ++k) c = (c >> 1) ^ ((c & 1) ? 0x82F63B78u : 0u);
            g_crc_tab[0][i] = c;
        }
        for (unsigned i = 0; i < 256; ++i)
            for (int t = 1; t < 8; ++t) g_crc_tab[t][i] = (g_crc_tab[t - 1][i] >> 8) ^ g_crc_tab[0][g_crc_tab[t - 1][i] & 0xff];
        g_crc_init = true;
    }
    const unsigned char* p = (const unsigned char*)data;
    crc ^= 0xffffffffu;
    while (n >= 8) {
        const unsigned lo = crc ^ ((unsigned)p[0] | ((unsigned)p[1] << 8) | ((unsigned)p[2] << 16) | ((unsigned)p[3] << 24));
        const unsigned hi = (unsigned)p[4] | ((unsigned)p[5] << 8) | ((unsigned)p[6] << 16) | ((unsigned)p[7] << 24);
        crc = g_crc_tab[7][lo & 0xff] ^ g_crc_tab[6][(lo >> 8) & 0xff] ^ g_crc_tab[5][(lo >> 16) & 0xff] ^ g_crc_tab[4][lo >> 24] ^
              g_crc_tab[3][hi & 0xff] ^ g_crc_tab[2][(hi >> 8) & 0xff] ^ g_crc_tab[1][(hi >> 16) & 0xff] ^ g_crc_tab[0][hi >> 24];
        p += 8;
        n -= 8;
    }
    while (n--) crc = g_crc_tab[0][(crc ^ *p++) & 0xff] ^ (crc >> 8);
    return crc ^ 0xffffffffu;
}

static std::atomic<long long> g_launches{0};
void atvs_count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }
extern "C" long long atvs_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int atvs_current_device(int* dev) {
    ATVS_CUDA(cudaGetDevice(dev));
    ATVS_CHECK_ARG(*dev >= 0 && *dev < ATVS_MAX_DEVICES, ATVS_E_UNSUP, "device %d: the library keeps state for devices "
                   "0..%d", *dev, ATVS_MAX_DEVICES - 1);
    return 0;
}

static std::atomic<int> g_sms[ATVS_MAX_DEVICES];
int atvs_num_sms() {
    int dev = 0;
    if (atvs_current_device(&dev) != 0) return 148;
    int n = g_sms[dev].load(std::memory_order_relaxed);
    if (n == 0) {
        if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
        g_sms[dev].store(n, std::memory_order_relaxed);
    }
    return n;
}

// per device: how many independent passes the caller runs side by side on its streams (pipeline.run_multiview); the
// plane-ring kernels size their grids with it (ring_common.cuh ring_balanced_grid).  0 = never set = 1.
static std::atomic<int> g_concurrency[ATVS_MAX_DEVICES];
int atvs_concurrency() {
    int dev = 0;
    if (atvs_current_device(&dev) != 0) return 1;
    const int n = g_concurrency[dev].load(std::memory_order_relaxed);
    return n < 1 ? 1 : n;
}
extern "C" int atvs_set_concurrency(int n) {
    int dev = 0;
    if (const int rc = atvs_current_device(&dev)) return rc;
    g_concurrency[dev].store(n < 1 ? 1 : (n > 64 ? 64 : n), std::memory_order_relaxed);
    return 0;
}

static unsigned long long* g_sat[ATVS_MAX_DEVICES] = {nullptr};
unsigned long long* atvs_sat_ptr() {
    int dev = 0;
    if (atvs_current_device(&dev) != 0) return nullptr;
    if (g_sat[dev] == nullptr) {
        unsigned long long* p = nullptr;
        if (cudaMalloc(&p, sizeof(unsigned long long)) != cudaSuccess) { cudaGetLastError(); return nullptr; }
        cudaMemset(p, 0, sizeof(unsigned long long));
        g_sat[dev] = p;
    }
    return g_sat[dev];
}
extern "C" long long atvs_saturation_count(int reset) {
    unsigned long long* p = atvs_sat_ptr();
    if (p == nullptr) return -1;
    unsigned long long v = 0;
    if (cudaMemcpy(&v, p, sizeof(v), cudaMemcpyDeviceToHost) != cudaSuccess) return -1;     // synchronises the device
    if (reset) cudaMemset(p, 0, sizeof(v));
    return (long long)v;
}
