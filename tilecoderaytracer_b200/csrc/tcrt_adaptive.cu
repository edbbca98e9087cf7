// tcrt_adaptive.cu — adaptive anti-aliasing (tcrt_render_columns_adaptive): the edge mask of a plain frame, the list of
// the pixels it marks, and the resolve of their samples.
//
// A frame is P (the plain frame) where a pixel's 3x3 neighbourhood shows no contrast, and the supersampled pixel of
// tcrt_render_columns_ss where it does (the contract is in include/tcrt.h).  The host renders P over the band plus one
// halo column on each side, then:
//   classify   one thread per band pixel, z fastest: quant8 of the pixel and its in-frame neighbours, the mask byte, P
//              copied into the band's frame; per CTA the number of marked pixels;
//   scan       one CTA: exclusive scan of those counts, total at the end (the model is the .txt formatter's two-level
//              scan, tcrt_format.cu);
//   compact    the marked pixels' x*H + z, in x-major order, at their scanned positions: a stable compaction, so the list
//              and everything sized or cut from it is deterministic;
// and, after the render kernels' list mode has traced samples 1 .. ss*ss-1 of a piece of the list into scratch,
//   resolve    one thread per list entry: acc = the frame pixel (sample (0,0) is the plain pixel, bit for bit), += the
//              other samples in tcrt.h's order, / (float)(ss*ss), back into the frame.
#include "tcrt_device.h"

namespace {

constexpr int kAdBlock = 256;

// quant8 of tcrt_format.cu: floor(clamp(c, 0, 1) * 255 + 0.5) on the float promoted to double, NaN -> 0
__device__ __forceinline__ int quant8(float v) {
    const double c = (double)v;
    const double cl = c > 0.0 ? (c < 1.0 ? c : 1.0) : 0.0;
    return (int)floor(cl * 255.0 + 0.5);
}

// plain: columns [px0, px0 + pcols) of the W x H frame, x-major, covering [bx0 - 1, bx1 + 1) clipped to [0, W).
__global__ void __launch_bounds__(kAdBlock) classify_kernel(const float* __restrict__ plain, int px0, int W, int H, int bx0,
                                                            int bx1, int contrast, float* __restrict__ frame,
                                                            unsigned char* __restrict__ mask, unsigned int* __restrict__ block_counts) {
    __shared__ unsigned int warp_cnt[kAdBlock / 32];
    const long long n = (long long)(bx1 - bx0) * H;
    const long long p = blockIdx.x * (long long)kAdBlock + threadIdx.x;
    bool refined = false;
    if (p < n) {
        const int xb = (int)(p / H), z = (int)(p - (long long)xb * H);
        const int x = bx0 + xb;
        const float* c = plain + ((size_t)(x - px0) * H + z) * 3;
        const float r = c[0], g = c[1], b = c[2];
        refined = contrast < 0;
        if (!refined) {
            const int q0 = quant8(r), q1 = quant8(g), q2 = quant8(b);
            for (int dx = -1; dx <= 1; ++dx) {
                const int xn = x + dx;
                if (xn < 0 || xn >= W) continue;
                for (int dz = -1; dz <= 1; ++dz) {
                    const int zn = z + dz;
                    if (zn < 0 || zn >= H || (dx == 0 && dz == 0)) continue;
                    const float* o = plain + ((size_t)(xn - px0) * H + zn) * 3;
                    const int d = max(abs(quant8(o[0]) - q0), max(abs(quant8(o[1]) - q1), abs(quant8(o[2]) - q2)));
                    refined = refined || d > contrast;
                }
            }
        }
        float* f = frame + (size_t)p * 3;
        f[0] = r;
        f[1] = g;
        f[2] = b;
        mask[p] = refined ? 1 : 0;
    }
    const unsigned int wc = __popc(__ballot_sync(0xffffffffu, refined));
    if ((threadIdx.x & 31) == 0) warp_cnt[threadIdx.x >> 5] = wc;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int t = 0;
        for (int w = 0; w < kAdBlock / 32; ++w) t += warp_cnt[w];
        block_counts[blockIdx.x] = t;
    }
}

// single CTA: exclusive scan of counts[0, n) in place, total at counts[n]
__global__ void __launch_bounds__(1024) scan_kernel(unsigned int* counts, int n) {
    __shared__ unsigned int warp_tot[32];
    __shared__ unsigned int carry;
    if (threadIdx.x == 0) carry = 0;
    __syncthreads();
    for (int i0 = 0; i0 < n; i0 += 1024) {
        const int i = i0 + (int)threadIdx.x;
        const unsigned int v = i < n ? counts[i] : 0u;
        unsigned int incl = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned int t = __shfl_up_sync(0xffffffffu, incl, o);
            if ((threadIdx.x & 31) >= (unsigned)o) incl += t;
        }
        if ((threadIdx.x & 31) == 31) warp_tot[threadIdx.x >> 5] = incl;
        __syncthreads();
        unsigned int base = carry;
        for (int w = 0; w < (int)(threadIdx.x >> 5); ++w) base += warp_tot[w];
        if (i < n) counts[i] = base + incl - v;
        __syncthreads();
        if (threadIdx.x == 1023) carry = base + incl;
        __syncthreads();
    }
    if (threadIdx.x == 0) counts[n] = carry;
}

// the marked pixels of the band, x*H + z of the frame, in band order at list[block offset + rank in the CTA]
__global__ void __launch_bounds__(kAdBlock) compact_kernel(const unsigned char* __restrict__ mask, int H, int bx0, int bx1,
                                                           const unsigned int* __restrict__ block_offs, int* __restrict__ list) {
    __shared__ unsigned int warp_cnt[kAdBlock / 32];
    const long long n = (long long)(bx1 - bx0) * H;
    const long long p = blockIdx.x * (long long)kAdBlock + threadIdx.x;
    const bool refined = p < n && mask[p] != 0;
    const unsigned int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const unsigned int bal = __ballot_sync(0xffffffffu, refined);
    if (lane == 0) warp_cnt[w] = __popc(bal);
    __syncthreads();
    if (refined) {
        unsigned int off = block_offs[blockIdx.x] + __popc(bal & ((1u << lane) - 1u));
        for (unsigned int k = 0; k < w; ++k) off += warp_cnt[k];
        list[off] = (int)(p + (long long)bx0 * H);   // (bx0 + xb) * H + z
    }
}

// entries [e0, e0 + n) of the list: samples 1 .. SS*SS-1 of entry e0 + t at scratch[(t*(SS*SS-1) + s-1)*3 ..]
template <int SS>
__global__ void __launch_bounds__(kAdBlock) resolve_list_kernel(const int* __restrict__ list, int e0, int n, int bx0, int H,
                                                                const float* __restrict__ scratch, float* __restrict__ frame) {
    constexpr int M = SS * SS - 1;
    const int t = blockIdx.x * kAdBlock + threadIdx.x;
    if (t >= n) return;
    const size_t px = (size_t)(__ldg(list + e0 + t) - bx0 * H);   // pixel of the band
    float* f = frame + px * 3;
    float acc[3] = {f[0], f[1], f[2]};                            // sample (0,0): the plain pixel
    const float* s = scratch + (size_t)t * M * 3;
#pragma unroll
    for (int k = 0; k < M; ++k)
#pragma unroll
        for (int c = 0; c < 3; ++c) acc[c] = __fadd_rn(acc[c], __ldg(s + 3 * k + c));
#pragma unroll
    for (int c = 0; c < 3; ++c) f[c] = __fdiv_rn(acc[c], (float)(SS * SS));
}

}  // namespace

cudaError_t tcrt_launch_adaptive_classify(const float* plain, int px0, int width, int height, int bx0, int bx1, int contrast,
                                          float* frame, unsigned char* mask, unsigned int* block_counts, int* list,
                                          cudaStream_t stream) {
    const long long n = (long long)(bx1 - bx0) * height;
    if (n <= 0) return cudaErrorInvalidValue;
    const int nb = (int)((n + kAdBlock - 1) / kAdBlock);
    classify_kernel<<<nb, kAdBlock, 0, stream>>>(plain, px0, width, height, bx0, bx1, contrast, frame, mask, block_counts);
    scan_kernel<<<1, 1024, 0, stream>>>(block_counts, nb);
    compact_kernel<<<nb, kAdBlock, 0, stream>>>(mask, height, bx0, bx1, block_counts, list);
    return cudaGetLastError();
}

cudaError_t tcrt_launch_adaptive_resolve(const int* list, int e0, int n, int bx0, int height, int ss, const float* scratch,
                                         float* frame, cudaStream_t stream) {
    if (n <= 0) return cudaSuccess;
    const int grid = (n + kAdBlock - 1) / kAdBlock;
    switch (ss) {
        case 2: resolve_list_kernel<2><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 3: resolve_list_kernel<3><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 4: resolve_list_kernel<4><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 5: resolve_list_kernel<5><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 6: resolve_list_kernel<6><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 7: resolve_list_kernel<7><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        case 8: resolve_list_kernel<8><<<grid, kAdBlock, 0, stream>>>(list, e0, n, bx0, height, scratch, frame); break;
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}
