// tcrt_format.cu — the .txt writer's pixel lines on the GPU.
//
// Replaces the loop of printPixelsToLog (RayTracer.cpp:1589-1602):
//     sprintf(line_str, "(%f, %f, %f)\n", temp->r, temp->g, temp->b); fputs(line_str, log_file);
// Output is byte-identical to glibc's "%f" of the float promoted to double: the value is
// M * 2^E exactly (M < 2^24), so  round_half_even(M * 10^6 * 2^E)  is computed in integers
// (64-bit for E < 0; up to 128-bit for the integer part of huge values) — SURVEY §8a row W.
//
// Two paths:
//   fixed   every channel prints as "d.dddddd" (0 <= v, rounds below 10): each line is exactly
//           31 bytes.  A CTA formats 256 pixels into shared memory and streams the 7936 bytes
//           out as 16-byte vectors.  This is every scene probed so far (SURVEY §8d).
//   general variable line lengths (values >= 10, negatives, inf/nan): per-pixel lengths,
//           a two-level exclusive scan, then byte stores at the scanned offsets.
#include "tcrt_device.h"

#include <algorithm>

namespace {

constexpr int kFmtBlock = 256;
constexpr int kLineFixed = 31;

// round_half_even(|v| * 10^6) for |v| < 2^24 (E < 0 path); returns false when E >= 0.
__device__ __forceinline__ bool micro_units(unsigned int bits, unsigned long long& q) {
    unsigned int ex = (bits >> 23) & 0xffu;
    unsigned int man = bits & 0x7fffffu;
    unsigned int M = ex ? (man | 0x800000u) : man;
    int E = (int)(ex ? ex : 1u) - 150;
    if (E >= 0) return false;
    int s = -E;
    unsigned long long p = (unsigned long long)M * 1000000ull;   // < 2^44
    if (s >= 46) {
        q = 0;   // p < 2^44 <= 2^(s-2): below half a unit
        return true;
    }
    q = p >> s;
    unsigned long long rem = p & ((1ull << s) - 1ull);
    unsigned long long half = 1ull << (s - 1);
    if (rem > half || (rem == half && (q & 1ull))) ++q;
    return true;
}

// True when v prints as exactly 8 characters "d.dddddd".
__device__ __forceinline__ bool is_fixed8(float v, unsigned int& q_out) {
    unsigned int bits = __float_as_uint(v);
    if (bits >> 31) return false;                 // negatives (and -0) carry a sign
    if (((bits >> 23) & 0xffu) == 0xffu) return false;
    unsigned long long q;
    if (!micro_units(bits, q)) return false;
    if (q >= 10000000ull) return false;
    q_out = (unsigned int)q;
    return true;
}

__device__ __forceinline__ void put_fixed8(char* o, unsigned int q) {
    unsigned int ip = q / 1000000u;
    unsigned int fr = q - ip * 1000000u;
    o[0] = (char)('0' + ip);
    o[1] = '.';
#pragma unroll
    for (int k = 5; k >= 0; --k) {
        unsigned int d = fr / 10u;
        o[2 + k] = (char)('0' + (fr - d * 10u));
        fr = d;
    }
}

// General "%f": returns the length written to o (<= 47).
__device__ int put_general(char* o, float v) {
    unsigned int bits = __float_as_uint(v);
    int n = 0;
    if (bits >> 31) o[n++] = '-';
    unsigned int ex = (bits >> 23) & 0xffu;
    unsigned int man = bits & 0x7fffffu;
    if (ex == 0xffu) {
        const char* w = man ? "nan" : "inf";
        o[n++] = w[0]; o[n++] = w[1]; o[n++] = w[2];
        return n;
    }
    unsigned long long q;
    unsigned int frac = 0;
    char tmp[40];
    int k = 0;
    if (micro_units(bits, q)) {
        unsigned long long ip = q / 1000000ull;
        frac = (unsigned int)(q - ip * 1000000ull);
        do { tmp[k++] = (char)('0' + (int)(ip % 10ull)); ip /= 10ull; } while (ip);
    } else {
        unsigned int M = man | 0x800000u;
        int E = (int)ex - 150;
        if (E <= 40) {
            unsigned long long ip = (unsigned long long)M << E;
            do { tmp[k++] = (char)('0' + (int)(ip % 10ull)); ip /= 10ull; } while (ip);
        } else {
            unsigned __int128 ip = (unsigned __int128)M << E;
            do { tmp[k++] = (char)('0' + (int)(ip % 10)); ip /= 10; } while (ip);
        }
    }
    while (k > 0) o[n++] = tmp[--k];
    o[n++] = '.';
    for (int j = 5; j >= 0; --j) {
        unsigned int d = frac / 10u;
        o[n + j] = (char)('0' + (frac - d * 10u));
        frac = d;
    }
    return n + 6;
}

__device__ int line_general(char* o, float r, float g, float b) {
    int n = 0;
    o[n++] = '(';
    n += put_general(o + n, r);
    o[n++] = ','; o[n++] = ' ';
    n += put_general(o + n, g);
    o[n++] = ','; o[n++] = ' ';
    n += put_general(o + n, b);
    o[n++] = ')'; o[n++] = '\n';
    return n;
}

// ---- fixed path ------------------------------------------------------------------------------
__global__ void __launch_bounds__(kFmtBlock) txt_fixed_check_kernel(const float* __restrict__ rgb, size_t n_floats,
                                                                    unsigned int* not_fixed) {
    bool bad = false;
    for (size_t i = blockIdx.x * (size_t)kFmtBlock + threadIdx.x; i < n_floats; i += (size_t)gridDim.x * kFmtBlock) {
        unsigned int q;
        if (!is_fixed8(rgb[i], q)) bad = true;
    }
    if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicOr(not_fixed, 1u);
}

__global__ void __launch_bounds__(kFmtBlock) txt_fixed_kernel(const float* __restrict__ rgb, size_t n_pixels,
                                                              char* __restrict__ text) {
    __shared__ __align__(16) char stage[kFmtBlock * kLineFixed];   // 7936 B = 496 x 16 B
    __shared__ float in[kFmtBlock * 3];
    const size_t n_tiles = (n_pixels + kFmtBlock - 1) / kFmtBlock;
    for (size_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const size_t p0 = tile * kFmtBlock;
        const int np = (int)min((size_t)kFmtBlock, n_pixels - p0);
        // coalesced load of np*3 floats
        for (int i = threadIdx.x; i < np * 3; i += kFmtBlock) in[i] = rgb[p0 * 3 + i];
        __syncthreads();
        if ((int)threadIdx.x < np) {
            char* o = stage + threadIdx.x * kLineFixed;
            unsigned int q0 = 0, q1 = 0, q2 = 0;
            is_fixed8(in[3 * threadIdx.x + 0], q0);
            is_fixed8(in[3 * threadIdx.x + 1], q1);
            is_fixed8(in[3 * threadIdx.x + 2], q2);
            o[0] = '(';
            put_fixed8(o + 1, q0);
            o[9] = ','; o[10] = ' ';
            put_fixed8(o + 11, q1);
            o[19] = ','; o[20] = ' ';
            put_fixed8(o + 21, q2);
            o[29] = ')'; o[30] = '\n';
        }
        __syncthreads();
        const size_t byte0 = p0 * kLineFixed;      // multiple of 7936 -> 16-byte aligned
        const int nbytes = np * kLineFixed;
        const int nvec = nbytes / 16;
        uint4* dst = reinterpret_cast<uint4*>(text + byte0);
        const uint4* src = reinterpret_cast<const uint4*>(stage);
        for (int i = threadIdx.x; i < nvec; i += kFmtBlock) dst[i] = src[i];
        for (int i = nvec * 16 + threadIdx.x; i < nbytes; i += kFmtBlock) text[byte0 + i] = stage[i];
        __syncthreads();
    }
}

// ---- general path ------------------------------------------------------------------------------
// offs[i] = exclusive prefix of line lengths inside the tile; block_sums[tile] = tile total.
__global__ void __launch_bounds__(kFmtBlock) txt_len_kernel(const float* __restrict__ rgb, size_t n_pixels,
                                                            unsigned long long* __restrict__ offs,
                                                            unsigned long long* __restrict__ block_sums) {
    __shared__ unsigned int warp_tot[kFmtBlock / 32];
    const size_t p = blockIdx.x * (size_t)kFmtBlock + threadIdx.x;
    char scratch[160];
    unsigned int len = 0;
    if (p < n_pixels) len = (unsigned int)line_general(scratch, rgb[3 * p], rgb[3 * p + 1], rgb[3 * p + 2]);
    unsigned int incl = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
        if ((threadIdx.x & 31) >= o) incl += t;
    }
    if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
    __syncthreads();
    unsigned int base = 0;
    for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) base += warp_tot[w];
    if (p < n_pixels) offs[p] = (unsigned long long)(base + incl - len);
    if (threadIdx.x == kFmtBlock - 1) block_sums[blockIdx.x] = (unsigned long long)(base + incl);
}

// single CTA: exclusive scan of block_sums in place; total appended at block_sums[n]
__global__ void __launch_bounds__(1024) txt_scan_kernel(unsigned long long* block_sums, size_t n) {
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (size_t i0 = 0; i0 < n; i0 += 1024) {
        size_t i = i0 + threadIdx.x;
        unsigned long long v = (i < n) ? block_sums[i] : 0ull;
        unsigned long long incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
        __syncthreads();
        unsigned long long base = carry;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) base += warp_tot[w];
        if (i < n) block_sums[i] = base + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = base + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) block_sums[n] = carry;
}

__global__ void __launch_bounds__(kFmtBlock) txt_general_kernel(const float* __restrict__ rgb, size_t n_pixels,
                                                                const unsigned long long* __restrict__ offs,
                                                                const unsigned long long* __restrict__ block_offs,
                                                                char* __restrict__ text) {
    const size_t p = blockIdx.x * (size_t)kFmtBlock + threadIdx.x;
    if (p >= n_pixels) return;
    char line[160];
    int n = line_general(line, rgb[3 * p], rgb[3 * p + 1], rgb[3 * p + 2]);
    char* o = text + block_offs[blockIdx.x] + offs[p];
    for (int i = 0; i < n; ++i) o[i] = line[i];
}

__global__ void l2_flush_kernel(uint4* p, size_t n) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        p[i] = make_uint4(0u, 1u, 2u, 3u);
}

}  // namespace

cudaError_t tcrt_launch_txt_fixed_check(const float* rgb, size_t n_pixels, unsigned int* not_fixed_flag,
                                        cudaStream_t stream) {
    if (n_pixels == 0) return cudaSuccess;
    txt_fixed_check_kernel<<<148 * 8, kFmtBlock, 0, stream>>>(rgb, n_pixels * 3, not_fixed_flag);
    return cudaGetLastError();
}

cudaError_t tcrt_launch_txt_fixed(const float* rgb, size_t n_pixels, char* text, cudaStream_t stream) {
    if (n_pixels == 0) return cudaSuccess;
    size_t tiles = (n_pixels + kFmtBlock - 1) / kFmtBlock;
    int grid = (int)min(tiles, (size_t)148 * 8);
    txt_fixed_kernel<<<grid, kFmtBlock, 0, stream>>>(rgb, n_pixels, text);
    return cudaGetLastError();
}

// offs: n_pixels uint64; block_sums: ceil(n_pixels/256) + 1 uint64.  After this,
// block_sums[0..nb) are exclusive tile offsets and block_sums[nb] the total byte count.
cudaError_t tcrt_launch_txt_lengths(const float* rgb, size_t n_pixels, unsigned long long* offs,
                                    unsigned long long* block_sums, cudaStream_t stream, int* launches) {
    if (n_pixels == 0) return cudaSuccess;
    size_t nb = (n_pixels + kFmtBlock - 1) / kFmtBlock;
    txt_len_kernel<<<(unsigned)nb, kFmtBlock, 0, stream>>>(rgb, n_pixels, offs, block_sums);
    txt_scan_kernel<<<1, 1024, 0, stream>>>(block_sums, nb);
    if (launches) *launches += 2;
    return cudaGetLastError();
}

cudaError_t tcrt_launch_txt_general(const float* rgb, size_t n_pixels, const unsigned long long* offs,
                                     const unsigned long long* block_offs, char* text, cudaStream_t stream) {
    if (n_pixels == 0) return cudaSuccess;
    size_t nb = (n_pixels + kFmtBlock - 1) / kFmtBlock;
    txt_general_kernel<<<(unsigned)nb, kFmtBlock, 0, stream>>>(rgb, n_pixels, offs, block_offs, text);
    return cudaGetLastError();
}

cudaError_t tcrt_launch_l2_flush(void* scratch, size_t bytes, cudaStream_t stream) {
    l2_flush_kernel<<<148 * 4, 256, 0, stream>>>(reinterpret_cast<uint4*>(scratch), bytes / 16);
    return cudaGetLastError();
}

// ---- FP32 pipe microbenchmark (roofline denominator) -------------------------------------------
namespace {
template <bool FMA>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float m, float c) {
    float a[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) a[k] = (float)(threadIdx.x + k) * 1e-3f;
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (FMA) a[k] = __fmaf_rn(a[k], m, c);
            else a[k] = __fadd_rn(__fmul_rn(a[k], m), c);
        }
    }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) s += a[k];
    if (s == 123.456f) out[0] = s;   // keep the chains alive
}
}  // namespace

cudaError_t tcrt_launch_fp32_peak(bool fma, float* scratch, int grid, int iters, cudaStream_t stream) {
    if (fma) fp32_peak_kernel<true><<<grid, 256, 0, stream>>>(scratch, iters, 0.999f, 1e-3f);
    else fp32_peak_kernel<false><<<grid, 256, 0, stream>>>(scratch, iters, 0.999f, 1e-3f);
    return cudaGetLastError();
}

// ---- 8-bit quantisation for the image outputs (tcrt_write_ppm) ------------------------------------------
// q(c) = floor(clamp(c, 0, 1) * 255 + 0.5) on the float promoted to double: the quantisation the
// parity tolerance is stated in (SURVEY §8a, last row).  NaN -> 0.  The kernel also turns the x-major band
// (column by column, z up) into image rows (top row first): a 32x32-pixel tile goes through shared memory, so
// both the float reads (along z) and the byte writes (along x) are contiguous.
namespace {
__device__ __forceinline__ unsigned char quant8(float v) {
    const double c = (double)v;
    const double cl = c > 0.0 ? (c < 1.0 ? c : 1.0) : 0.0;   // NaN fails both compares -> 0
    return (unsigned char)floor(cl * 255.0 + 0.5);
}
// rgb: cols x height pixels, x-major.  out: height rows of cols pixels, row 0 = z = height-1.
__global__ void __launch_bounds__(256) quantize8_image_kernel(const float* __restrict__ rgb, int cols, int height,
                                                              unsigned char* __restrict__ out) {
    __shared__ unsigned char tile[32][32 * 3 + 1];     // [x in tile][z in tile][channel]
    const int tiles_z = (height + 31) / 32, tiles_x = (cols + 31) / 32;
    for (int t = blockIdx.x; t < tiles_x * tiles_z; t += gridDim.x) {
        const int x0 = (t / tiles_z) * 32, z0 = (t % tiles_z) * 32;
        for (int i = threadIdx.x; i < 32 * 96; i += 256) {       // 32 columns x (32 rows x 3 channels), contiguous along z
            const int xx = i / 96, k = i % 96;
            const int x = x0 + xx, z = z0 + k / 3;
            if (x < cols && z < height) tile[xx][k] = quant8(rgb[((size_t)x * height + z0) * 3 + k]);
        }
        __syncthreads();
        for (int i = threadIdx.x; i < 32 * 96; i += 256) {       // 32 rows x (32 columns x 3 channels), contiguous along x
            const int zz = i / 96, k = i % 96;
            const int z = z0 + zz, x = x0 + k / 3;
            if (x < cols && z < height) out[((size_t)(height - 1 - z) * cols + x0) * 3 + k] = tile[k / 3][zz * 3 + k % 3];
        }
        __syncthreads();
    }
}
}  // namespace

// Element-wise q(c) of a run of floats into as many bytes: float j -> byte j, so an x-major band stays x-major (3 bytes a
// pixel).  `head` scalar elements bring rgb to 16 bytes and out to 4 bytes; the body is one float4 in, one u32 out per
// thread and step; the rest is the scalar tail.
__global__ void __launch_bounds__(256) tcrt_quantize8_kernel(const float* __restrict__ rgb, size_t n, size_t head,
                                                             size_t n_vec, unsigned char* __restrict__ out) {
    const size_t tid = blockIdx.x * (size_t)blockDim.x + threadIdx.x, stride = (size_t)gridDim.x * blockDim.x;
    const float4* in4 = reinterpret_cast<const float4*>(rgb + head);
    unsigned int* out4 = reinterpret_cast<unsigned int*>(out + head);
    for (size_t i = tid; i < n_vec; i += stride) {
        const float4 v = in4[i];
        out4[i] = (unsigned int)quant8(v.x) | (unsigned int)quant8(v.y) << 8 | (unsigned int)quant8(v.z) << 16 |
                  (unsigned int)quant8(v.w) << 24;
    }
    const size_t tail0 = head + 4 * n_vec;
    for (size_t i = tid; i < head + (n - tail0); i += stride) {
        const size_t j = i < head ? i : tail0 + (i - head);
        out[j] = quant8(rgb[j]);
    }
}

cudaError_t tcrt_launch_quantize8(const float* rgb, size_t n_pixels, unsigned char* out, cudaStream_t stream) {
    if (n_pixels == 0) return cudaSuccess;
    const size_t n = 3 * n_pixels;
    // the first element at which both pointers are aligned; a pair that never is (not the case of the frame buffers,
    // which sit at the same pixel offset of two cudaMalloc blocks) takes the scalar loop alone
    size_t head = n, n_vec = 0;
    for (size_t h = 0; h < 4 && h < n; h++)
        if (((uintptr_t)(rgb + h) & 15) == 0 && ((uintptr_t)(out + h) & 3) == 0) {
            head = h;
            n_vec = (n - h) / 4;
            break;
        }
    const size_t work = std::max(n_vec, head + (n - head - 4 * n_vec));
    const int grid = (int)std::min<size_t>((work + 255) / 256, (size_t)148 * 8);
    tcrt_quantize8_kernel<<<grid, 256, 0, stream>>>(rgb, n, head, n_vec, out);
    return cudaGetLastError();
}

// ---- supersampled frames: the box filter over SS x SS samples per pixel -------------------------------------------------
// samples: SS*cols sample columns of SS*height sample rows, x-major; sample (i, j) of output pixel (x, z) is sample pixel
// (SS*x + i, SS*z + j).  For fixed i the SS samples of a pixel are one run of 3*SS contiguous floats, and the run of pixel
// z+1 follows it: one thread per output pixel with z fastest makes a warp read 32 consecutive runs.  The runs are loaded
// as float4 (SS % 4 == 0) or float2 (SS even) — every run and every sample column then starts at a multiple of that
// width — and as floats otherwise.  The sum is the contract of tcrt_render_columns_ss: acc = sample (0,0), then += in
// i-major, j-minor order, then one IEEE division by SS*SS.  out8 (optional) gets quant8 of the resolved floats.
namespace {
template <int SS>
__global__ void __launch_bounds__(256) resolve_ss_kernel(const float* __restrict__ samples, int cols, int height,
                                                         float* __restrict__ out, unsigned char* __restrict__ out8) {
    constexpr int V = SS % 4 == 0 ? 4 : (SS % 2 == 0 ? 2 : 1);     // floats per load
    constexpr int R = 3 * SS;                                      // floats per run
    const long long px = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (px >= (long long)cols * height) return;
    const int x = (int)(px / height), z = (int)(px - (long long)x * height);
    const size_t col = (size_t)SS * height * 3;                    // floats per sample column
    const float* s = samples + (size_t)SS * x * col + (size_t)R * z;
    float acc[3] = {0.f, 0.f, 0.f};    // set to sample (0,0) below
#pragma unroll
    for (int i = 0; i < SS; i++) {
        float run[R];
#pragma unroll
        for (int k = 0; k < R; k += V) {
            if constexpr (V == 4) {
                const float4 v = __ldg(reinterpret_cast<const float4*>(s + i * col + k));
                run[k] = v.x; run[k + 1] = v.y; run[k + 2] = v.z; run[k + 3] = v.w;
            } else if constexpr (V == 2) {
                const float2 v = __ldg(reinterpret_cast<const float2*>(s + i * col + k));
                run[k] = v.x; run[k + 1] = v.y;
            } else {
                run[k] = __ldg(s + i * col + k);
            }
        }
#pragma unroll
        for (int j = 0; j < SS; j++)
#pragma unroll
            for (int c = 0; c < 3; c++) acc[c] = (i == 0 && j == 0) ? run[c] : __fadd_rn(acc[c], run[3 * j + c]);
    }
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const float v = __fdiv_rn(acc[c], (float)(SS * SS));
        out[px * 3 + c] = v;
        if (out8) out8[px * 3 + c] = quant8(v);
    }
}
}  // namespace

cudaError_t tcrt_launch_resolve_ss(const float* samples, int cols, int height, int ss, float* out, unsigned char* out8,
                                   cudaStream_t stream) {
    if (cols <= 0 || height <= 0) return cudaSuccess;
    const int grid = (int)(((long long)cols * height + 255) / 256);
    switch (ss) {
        case 1: resolve_ss_kernel<1><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 2: resolve_ss_kernel<2><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 3: resolve_ss_kernel<3><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 4: resolve_ss_kernel<4><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 5: resolve_ss_kernel<5><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 6: resolve_ss_kernel<6><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 7: resolve_ss_kernel<7><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        case 8: resolve_ss_kernel<8><<<grid, 256, 0, stream>>>(samples, cols, height, out, out8); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

cudaError_t tcrt_launch_quantize8_image(const float* rgb, int cols, int height, unsigned char* out, cudaStream_t stream) {
    if (cols <= 0 || height <= 0) return cudaSuccess;
    const long long tiles = (long long)((cols + 31) / 32) * ((height + 31) / 32);
    quantize8_image_kernel<<<(int)min(tiles, (long long)148 * 8), 256, 0, stream>>>(rgb, cols, height, out);
    return cudaGetLastError();
}
