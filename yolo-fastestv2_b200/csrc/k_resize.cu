// Device-side cv2.resize(img, (W, H), interpolation=cv2.INTER_LINEAR) for uint8 BGR images (reference utils/datasets.py:106-111,
// test.py:34-37), fused with the HWC -> CHW transpose that follows it: a ragged batch of N HWC sources in, the NCHW uint8 batch
// yfv2_forward_u8 consumes out.  OpenCV's fixed-point arithmetic, reproduced bit for bit (oracle/resize.py states it):
//   columns  fx = fl32((dx + 0.5) * scale_x - 0.5), sx = floor(fx), fx -= sx, edge columns clamp sx and zero fx,
//            a0 = rint((1 - fx) * 2048), a1 = rint(fx * 2048)
//   rows     the same, but fy is not clamped (only the row indices are)
//   pass 1   T = src[r][sx] * a0 + src[r][sx + 1] * a1                                   (int32)
//   pass 2   out = sat_u8((((T0 >> 4) * b0 >> 16) + ((T1 >> 4) * b1 >> 16) + 2) >> 2)
// Every double / float operation below is written with an explicit _rn intrinsic so that nvcc cannot contract it into an FMA.
//
// One CTA per (image, band of B output rows).  The CTA builds the column table for its image in shared memory, works out which
// source rows its band reads (at most 2B; rows a downscale skips are never read), stages exactly those rows with 16-byte loads
// (cp.async) where the alignment allows and byte loads at the ragged edges (sources start at any byte), then computes 16 output
// bytes of one channel per work item and stores them as planar rows (16-byte stores when W and `out` allow it).  A staged row is
// shared by every output row of the band that reads it, which is what makes upscaling cheap.  Integer arithmetic only; the bound
// is HBM (rows read + output written), of which it reaches 0.16 so far (DESIGN.md §4).
#include "common.cuh"

namespace yfv2 {
namespace {

constexpr int kResizeMaxImages = 256;      // images per launch: their descriptors travel in the kernel parameters (3 KB)
constexpr int kResizeThreads = 256;
constexpr int kResizeMaxBand = 16;         // output rows per CTA
constexpr int kResizeRowBudget = 72 * 1024;  // shared memory for staged source rows

struct ResizeArgs {
    const uint8_t* src[kResizeMaxImages];
    unsigned hw[kResizeMaxImages];         // h << 16 | w
    uint8_t* out;                          // [n, 3, H, W] of this launch
    int H, W, band, rowstride;             // rowstride: bytes per staged row slot (multiple of 16)
    int vec16;                             // out rows are 16-byte aligned and W % 16 == 0
};

// Source coordinate of destination coordinate d: (floor, fractional part), exactly as OpenCV computes them.
__device__ __forceinline__ void resize_coord(int d, double scale, int& s, float& f) {
    const float fr = __double2float_rn(__dsub_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), 0.5));
    const float fl = floorf(fr);
    s = (int)fl;
    f = __fsub_rn(fr, fl);
}
__device__ __forceinline__ int coef0(float f) { return (int)rintf(__fmul_rn(__fsub_rn(1.f, f), 2048.f)); }
__device__ __forceinline__ int coef1(float f) { return (int)rintf(__fmul_rn(f, 2048.f)); }

__global__ void __launch_bounds__(kResizeThreads)
resize_linear_u8_kernel(const __grid_constant__ ResizeArgs a) {
    extern __shared__ __align__(16) uint8_t smem[];
    const int n = blockIdx.y;
    const int h = (int)(a.hw[n] >> 16), w = (int)(a.hw[n] & 0xffffu);
    const int H = a.H, W = a.W;
    const int y0 = blockIdx.x * a.band;
    const int nb = min(a.band, H - y0);
    const uint8_t* __restrict__ src = a.src[n];
    uint8_t* rows = smem;                                                     // 2 * band slots of rowstride bytes
    int4* rowtab = reinterpret_cast<int4*>(smem + 2 * a.band * a.rowstride);   // band: (row r0 byte offset, r1 offset, b0, b1)
    int* srow = reinterpret_cast<int*>(rowtab + a.band);                       // 2 * band: source row held by each slot
    uint2* coltab = reinterpret_cast<uint2*>(srow + 2 * a.band);               // 16 x groups: (3*sx0 | 3*sx1 << 16, a0 | a1 << 16)
    __shared__ int nslots;
    __shared__ int s_sy[kResizeMaxBand];
    __shared__ float s_fy[kResizeMaxBand];

    if (threadIdx.x < nb) {                              // row coordinates of the band, one thread per output row
        int sy; float fy;
        resize_coord(y0 + threadIdx.x, __drcp_rn(__ddiv_rn((double)H, (double)h)), sy, fy);
        s_sy[threadIdx.x] = sy;
        s_fy[threadIdx.x] = fy;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        // the source rows the band reads, each once: r0 and r1 never decrease with dy, so a row is one of the last two slots or new
        int k = 0;
        for (int i = 0; i < nb; ++i) {
            const int sy = s_sy[i];
            const int r[2] = {min(max(sy, 0), h - 1), min(max(sy + 1, 0), h - 1)};
            int slot[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                int q = k - 1;
                if (q >= 0 && srow[q] != r[j]) q = (q >= 1 && srow[q - 1] == r[j]) ? q - 1 : -1;
                if (q < 0) { q = k; srow[k++] = r[j]; }
                slot[j] = q * a.rowstride + (int)(reinterpret_cast<uintptr_t>(src + (size_t)r[j] * 3 * w) & 15);
            }
            rowtab[i] = make_int4(slot[0], slot[1], coef0(s_fy[i]), coef1(s_fy[i]));
        }
        nslots = k;
    }
    __syncthreads();

    // stage the rows: slot byte j holds global byte (row start rounded down to 16) + j, so the middle of a row moves in 16-byte
    // cp.async copies (all in flight at once, no register staging) and only the two ragged edge chunks byte by byte
    const int rb = 3 * w;
    const int chunks = (rb + 15) / 16 + 1;
    for (int t = threadIdx.x; t < nslots * chunks; t += blockDim.x) {
        const int k = t / chunks, c = t - k * chunks;
        const uint8_t* base = src + (size_t)srow[k] * rb;
        const uintptr_t lo = reinterpret_cast<uintptr_t>(base), hi = lo + rb;
        const uintptr_t g = (lo & ~(uintptr_t)15) + 16 * (uintptr_t)c;
        uint8_t* d = rows + k * a.rowstride + 16 * c;
        if (g >= lo && g + 16 <= hi) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"((unsigned)__cvta_generic_to_shared(d)), "l"(g) : "memory");
        } else {                                          // all 16 byte loads issued before the first store: one latency, not 16
            uint8_t v[16];
#pragma unroll
            for (int b = 0; b < 16; ++b)
                v[b] = (g + b >= lo && g + b < hi) ? __ldg(reinterpret_cast<const uint8_t*>(g + b)) : (uint8_t)0;
#pragma unroll
            for (int b = 0; b < 16; ++b)
                if (g + b >= lo && g + b < hi) d[b] = v[b];
        }
    }
    asm volatile("cp.async.commit_group;\n" ::: "memory");

    // the column table, while the rows are in flight; column 16*g + e at [e][g]: the lanes of a warp (consecutive g) read
    // consecutive entries for each e, where a column-major table put all 32 lanes of a warp in one bank
    const int groups = (W + 15) / 16;
    const double scale_x = __drcp_rn(__ddiv_rn((double)W, (double)w));
    for (int dx = threadIdx.x; dx < W; dx += blockDim.x) {
        int sx; float fx;
        resize_coord(dx, scale_x, sx, fx);
        if (sx < 0) { sx = 0; fx = 0.f; }
        if (sx >= w - 1) { sx = w - 1; fx = 0.f; }
        const int sx1 = min(sx + 1, w - 1);
        coltab[(dx & 15) * groups + (dx >> 4)] = make_uint2((unsigned)(3 * sx) | ((unsigned)(3 * sx1) << 16),
                                                            (unsigned)coef0(fx) | ((unsigned)coef1(fx) << 16));
    }
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
    __syncthreads();

    // compute: one work item = 16 consecutive output bytes of one channel of one output row
    for (int t = threadIdx.x; t < nb * 3 * groups; t += blockDim.x) {
        const int i = t / (3 * groups);
        const int rem = t - i * 3 * groups;
        const int ch = rem / groups, gx = rem - ch * groups;
        const int4 rt = rowtab[i];
        const uint8_t* q0 = rows + rt.x + ch;
        const uint8_t* q1 = rows + rt.y + ch;
        unsigned v[4] = {0u, 0u, 0u, 0u};
        const int x0 = 16 * gx, xe = min(16, W - x0);
#pragma unroll
        for (int e = 0; e < 16; ++e) {
            if (e < xe) {
                const uint2 ct = coltab[e * groups + gx];
                const int i0 = (int)(ct.x & 0xffffu), i1 = (int)(ct.x >> 16);
                const int c0 = (int)(ct.y & 0xffffu), c1 = (int)(ct.y >> 16);
                const int t0 = (int)q0[i0] * c0 + (int)q0[i1] * c1;
                const int t1 = (int)q1[i0] * c0 + (int)q1[i1] * c1;
                const int s = ((((t0 >> 4) * rt.z) >> 16) + (((t1 >> 4) * rt.w) >> 16) + 2) >> 2;
                v[e >> 2] |= (unsigned)min(max(s, 0), 255) << (8 * (e & 3));
            }
        }
        uint8_t* o = a.out + (((size_t)n * 3 + ch) * H + (y0 + i)) * (size_t)W + x0;
        if (a.vec16) {
            *reinterpret_cast<uint4*>(o) = make_uint4(v[0], v[1], v[2], v[3]);
        } else {
            for (int e = 0; e < xe; ++e) o[e] = (uint8_t)(v[e >> 2] >> (8 * (e & 3)));
        }
    }
}

}  // namespace
}  // namespace yfv2

extern "C" int yfv2_resize_u8(const uint8_t* const* src, const int* src_hw, int N, int H, int W, uint8_t* out, void* stream) {
    using namespace yfv2;
    if (!src || !src_hw || !out) { set_error("resize_u8: null pointer argument"); return YFV2_EINVAL; }
    if (N <= 0) { set_error("resize_u8: N = %d, need at least one image", N); return YFV2_EINVAL; }
    if (H <= 0 || W <= 0) { set_error("resize_u8: destination %d x %d is empty", H, W); return YFV2_EINVAL; }
    if (H > YFV2_RESIZE_MAX_DST || W > YFV2_RESIZE_MAX_DST) {
        set_error("resize_u8: destination %d x %d exceeds %d per side", H, W, YFV2_RESIZE_MAX_DST);
        return YFV2_EUNSUPPORTED;
    }
    const uintptr_t out_lo = reinterpret_cast<uintptr_t>(out), out_hi = out_lo + (uintptr_t)N * 3 * H * W;
    int wmax = 1;
    for (int i = 0; i < N; ++i) {
        const int h = src_hw[2 * i], w = src_hw[2 * i + 1];
        if (!src[i]) { set_error("resize_u8: source %d is a null pointer", i); return YFV2_EINVAL; }
        if (h <= 0 || w <= 0) { set_error("resize_u8: source %d is %d x %d", i, h, w); return YFV2_EINVAL; }
        if (h > YFV2_RESIZE_MAX_SRC || w > YFV2_RESIZE_MAX_SRC) {
            set_error("resize_u8: source %d is %d x %d, above %d per side", i, h, w, YFV2_RESIZE_MAX_SRC);
            return YFV2_EUNSUPPORTED;
        }
        const uintptr_t lo = reinterpret_cast<uintptr_t>(src[i]), hi = lo + (uintptr_t)3 * h * w;
        if (lo < out_hi && out_lo < hi) { set_error("resize_u8: out overlaps source %d", i); return YFV2_EINVAL; }
        wmax = w > wmax ? w : wmax;
    }
    const int rowstride = (3 * wmax + 15) / 16 * 16 + 16;
    int band = kResizeRowBudget / (2 * rowstride);
    band = band < 1 ? 1 : (band > kResizeMaxBand ? kResizeMaxBand : band);
    const size_t smem = (size_t)2 * band * rowstride + 24 * (size_t)band + 128 * (size_t)((W + 15) / 16);   // rows, rowtab + srow, coltab
    YFV2_CUDA(cudaFuncSetAttribute(resize_linear_u8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ResizeArgs a;
    a.H = H; a.W = W; a.band = band; a.rowstride = rowstride;
    for (int i0 = 0; i0 < N; i0 += kResizeMaxImages) {
        const int n = N - i0 < kResizeMaxImages ? N - i0 : kResizeMaxImages;
        for (int i = 0; i < n; ++i) {
            a.src[i] = src[i0 + i];
            a.hw[i] = ((unsigned)src_hw[2 * (i0 + i)] << 16) | (unsigned)src_hw[2 * (i0 + i) + 1];
        }
        a.out = out + (size_t)i0 * 3 * H * W;
        a.vec16 = (W % 16 == 0) && (reinterpret_cast<uintptr_t>(a.out) % 16 == 0);
        resize_linear_u8_kernel<<<dim3((unsigned)((H + band - 1) / band), (unsigned)n), kResizeThreads, smem, (cudaStream_t)stream>>>(a);
        YFV2_LAUNCH_CHECK();
    }
    return YFV2_OK;
}
