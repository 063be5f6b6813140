// C-ABI plumbing shared by every stage (error string, launch counter) plus the small
// data-movement stages: D0 image -> network input, and the stand-alone depth-to-space.
#include "common.cuh"
#include "../../include/balf_b200.h"

#include <string.h>
#include <string>
#include <vector>

namespace balf {

unsigned long long g_launches = 0;
static thread_local std::string g_error;

int set_error(int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_error = buf;
    return code;
}
const char* last_error() { return g_error.c_str(); }

// ---- per-kernel event timing
bool g_prof_on = false;
struct ProfRec { const char* name; cudaEvent_t e0, e1; };
static std::vector<ProfRec> g_prof;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t prof_event() {
    cudaEvent_t e;
    if (!g_prof_pool.empty()) { e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEventCreate(&e);
    return e;
}
void prof_begin(const char* name, cudaStream_t st) {
    ProfRec r{name, prof_event(), prof_event()};
    cudaEventRecord(r.e0, st);
    g_prof.push_back(r);
}
void prof_end(cudaStream_t st) { cudaEventRecord(g_prof.back().e1, st); }

// D0: demo_match.py:22-29.  float(u8) / 255.f is bit-identical to the reference's float64
// division followed by the fp32 cast for all 256 inputs (SURVEY.md section 8a, row D0).
__global__ void preprocess_u8_kernel(const uint8_t* __restrict__ img, int H, int W, int C, float* __restrict__ x,
                                     int Hp, int Wp, int top, int left) {
    // four output pixels per thread (Wp is a multiple of 64): one float4 store per plane
    const int xo = 4 * (blockIdx.x * blockDim.x + threadIdx.x), yo = blockIdx.y, b = blockIdx.z;
    if (xo >= Wp) return;
    const int yi = yo - top;
    const bool row_in = yi >= 0 && yi < H;
    float v[3][4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const int xi = xo + k - left;
        const bool in = row_in && xi >= 0 && xi < W;
        const uint8_t* px = img + (((size_t)b * H + (in ? yi : 0)) * W + (in ? xi : 0)) * C;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c][k] = in ? (float)px[C == 1 ? 0 : c] / 255.0f : 0.0f;
    }
#pragma unroll
    for (int c = 0; c < 3; ++c)
        *reinterpret_cast<float4*>(x + (((size_t)b * 3 + c) * Hp + yo) * Wp + xo) = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
}

// the byte-plane form of the same geometry for a gray image: g[b][yo][xo] = the image byte, 0 in the padding.  Sixteen output bytes
// per thread (Wp is a multiple of 16): one 16-byte store.
__global__ void pad_gray_u8_kernel(const uint8_t* __restrict__ img, int H, int W, uint8_t* __restrict__ g, int Hp, int Wp, int top,
                                   int left) {
    const int xo = 16 * (blockIdx.x * blockDim.x + threadIdx.x), yo = blockIdx.y, b = blockIdx.z;
    if (xo >= Wp) return;
    const int yi = yo - top;
    const bool row_in = yi >= 0 && yi < H;
    const uint8_t* src = img + ((size_t)b * H + (row_in ? yi : 0)) * W;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
#pragma unroll
    for (int k = 0; k < 16; ++k) {
        const int xi = xo + k - left;
        const uint32_t v = row_in && xi >= 0 && xi < W ? src[xi] : 0u;
        w[k / 4] |= v << (8 * (k % 4));
    }
    *reinterpret_cast<uint4*>(g + ((size_t)b * Hp + yo) * Wp + xo) = make_uint4(w[0], w[1], w[2], w[3]);
}

// tensor_op.py:1-27: out[n, c, r*i+a, r*j+b] = in[n, c*r*r + a*r + b, i, j]
__global__ void pixel_shuffle_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int H, int W, int r,
                                     size_t total) {
    size_t o = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (o >= total) return;
    const int Wo = W * r, Ho = H * r, Co = C / (r * r);
    int xo = (int)(o % Wo);
    size_t t = o / Wo;
    int yo = (int)(t % Ho);
    t /= Ho;
    int co = (int)(t % Co);
    size_t n = t / Co;
    int ci = co * r * r + (yo % r) * r + (xo % r);
    out[o] = in[((n * C + ci) * H + yo / r) * W + xo / r];
}

}  // namespace balf

using namespace balf;

extern "C" const char* balf_last_error(void) { return last_error(); }
extern "C" int balf_abi_version(void) { return BALF_B200_ABI_VERSION; }
extern "C" unsigned long long balf_launch_count(void) { return g_launches; }

extern "C" int balf_profile_enable(int on) {
    g_prof_on = on != 0;
    return 0;
}

// host-synchronous: waits for every recorded event, then writes "name count total_ms\n" lines
extern "C" int balf_profile_report(char* buf, size_t cap, int reset) {
    struct Agg { const char* name; long n; double ms; };
    std::vector<Agg> agg;
    for (ProfRec& r : g_prof) {
        BALF_CUDA_OK(cudaEventSynchronize(r.e1));
        float ms = 0.f;
        BALF_CUDA_OK(cudaEventElapsedTime(&ms, r.e0, r.e1));
        Agg* a = nullptr;
        for (Agg& q : agg) if (q.name == r.name || std::string(q.name) == r.name) { a = &q; break; }
        if (!a) { agg.push_back(Agg{r.name, 0, 0.0}); a = &agg.back(); }
        a->n += 1;
        a->ms += ms;
    }
    std::string out;
    char line[256];
    for (Agg& q : agg) {
        snprintf(line, sizeof(line), "%s %ld %.6f\n", q.name, q.n, q.ms);
        out += line;
    }
    if (buf && cap) {
        BALF_REQUIRE(out.size() + 1 <= cap, "profile report needs %zu bytes", out.size() + 1);
        memcpy(buf, out.c_str(), out.size() + 1);
    }
    if (reset) {
        for (ProfRec& r : g_prof) { g_prof_pool.push_back(r.e0); g_prof_pool.push_back(r.e1); }
        g_prof.clear();
    }
    return (int)out.size() + 1 > 0 ? 0 : 0;
}

extern "C" int balf_pad_geometry(int H, int W, int factor, int* Hp, int* Wp, int* top, int* left) {
    BALF_REQUIRE(H > 0 && W > 0 && factor > 0, "H, W, factor must be positive");
    // make_shape_even (test_utils.py:16-21) then mod_padding_symmetric (test_utils.py:23-32)
    const int he = H + (H & 1), we = W + (W & 1);
    const int ph = he % factor ? ((he + factor) / factor) * factor - he : 0;
    const int pw = we % factor ? ((we + factor) / factor) * factor - we : 0;
    if (Hp) *Hp = he + 2 * (ph / 2);
    if (Wp) *Wp = we + 2 * (pw / 2);
    if (top) *top = ph / 2;
    if (left) *left = pw / 2;
    return 0;
}

extern "C" int balf_preprocess_u8(const uint8_t* img, int B, int H, int W, int C, float* x, int Hp, int Wp, int top,
                                  int left, void* stream) {
    BALF_REQUIRE(img && x, "null pointer argument");
    BALF_REQUIRE(C == 1 || C == 3, "image must have 1 or 3 channels, got %d", C);
    BALF_REQUIRE(B > 0 && H > 0 && W > 0 && top >= 0 && left >= 0 && top + H <= Hp && left + W <= Wp,
                 "image %dx%d at (%d,%d) does not fit the padded size %dx%d", H, W, top, left, Hp, Wp);
    BALF_REQUIRE(Wp % 4 == 0, "padded width %d must be a multiple of 4", Wp);
    dim3 grid(cdiv(Wp, 4 * 128), Hp, B);
    {
        ProfScope p("preprocess_u8", static_cast<cudaStream_t>(stream));
        preprocess_u8_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(img, H, W, C, x, Hp, Wp, top, left);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}

extern "C" int balf_pad_gray_u8(const uint8_t* img, int B, int H, int W, uint8_t* g, int Hp, int Wp, int top, int left, void* stream) {
    BALF_REQUIRE(img && g, "null pointer argument");
    BALF_REQUIRE(B > 0 && H > 0 && W > 0 && top >= 0 && left >= 0 && top + H <= Hp && left + W <= Wp,
                 "image %dx%d at (%d,%d) does not fit the padded size %dx%d", H, W, top, left, Hp, Wp);
    BALF_REQUIRE(Hp % 64 == 0 && Wp % 64 == 0, "padded size %dx%d: height and width must be multiples of 64", Hp, Wp);
    dim3 grid(cdiv(Wp, 16 * 128), Hp, B);
    {
        ProfScope p("pad_gray_u8", static_cast<cudaStream_t>(stream));
        pad_gray_u8_kernel<<<grid, 128, 0, static_cast<cudaStream_t>(stream)>>>(img, H, W, g, Hp, Wp, top, left);
    }
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}

extern "C" int balf_pixel_shuffle(const float* in, float* out, int N, int C, int H, int W, int r, void* stream) {
    BALF_REQUIRE(in && out, "null pointer argument");
    BALF_REQUIRE(N > 0 && C > 0 && H > 0 && W > 0 && r > 0 && C % (r * r) == 0, "bad pixel_shuffle shape");
    size_t total = (size_t)N * C * H * W;
    pixel_shuffle_kernel<<<(unsigned)((total + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(in, out, C, H, W,
                                                                                                       r, total);
    BALF_COUNT_LAUNCH(1);
    BALF_LAUNCH_OK();
    return 0;
}
