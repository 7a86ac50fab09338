// tiles.cu - tile producer on the device (SURVEY §8 row n4).
// Test infrastructure it is not: this is the product path that replaces
// DOTA_devkit/SplitOnlyImage_multi_process.py:38-49 (saveimagepatches: crop subsize x subsize at (left, up), zero
// padded to the full tile) - the reference writes every tile to a PNG and the data loader decodes it again; here the
// decoded image is uploaded once and the batch of uint8 HWC tiles the detector consumes is cut out in HBM.
//
// The multi-scale producer (SplitOnlyImage_multi_process.py:53-58 resizes every image by cv2.resize INTER_CUBIC at rates
// 0.5 / 1.0 / 1.5 before cutting) computes each tile pixel straight from the original image with OpenCV's portable
// fixed-point bicubic arithmetic (DESIGN.md §2 deviation 7); the resized image is never materialised.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "common.cuh"

namespace orp {
namespace {

// one thread = 4 output bytes (out rows are subsize*C bytes, a multiple of 4 is required by the host wrapper)
__global__ void __launch_bounds__(256)
split_tiles_kernel(const uint8_t *__restrict__ img, int H, int W, int C, const int32_t *__restrict__ origins, int ntiles,
                   int subsize, uint8_t *__restrict__ out)
{
    const size_t row_bytes = (size_t)subsize * C;
    const size_t words_per_row = row_bytes / 4, words_per_tile = words_per_row * subsize;
    const size_t total = words_per_tile * ntiles;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int t = (int)(i / words_per_tile);
        const size_t r = i - (size_t)t * words_per_tile;
        const int y = (int)(r / words_per_row);
        const int xb = (int)(r - (size_t)y * words_per_row) * 4;           // byte offset inside the tile row
        const int left = origins[2 * t], up = origins[2 * t + 1];
        const int sy = up + y;
        const int valid_bytes = (W - left < subsize ? W - left : subsize) * C;   // bytes of this row that come from the image
        uint32_t v = 0;
        if (sy < H && xb < valid_bytes) {
            const uint8_t *src = img + ((size_t)sy * W + left) * C + xb;
#pragma unroll
            for (int k = 0; k < 4; ++k)
                if (xb + k < valid_bytes) v |= (uint32_t)src[k] << (8 * k);
        }
        reinterpret_cast<uint32_t *>(out)[i] = v;
    }
}

int grid_for(size_t items, int threads)
{
    size_t g = (items + threads - 1) / threads;
    const size_t cap = 148 * 16;
    return (int)(g < cap ? (g ? g : 1) : cap);
}

// ---- bicubic resize (cv2 INTER_CUBIC, fixed point: 11-bit weights per axis, int32 sums, rounding shift by 22) ----

// one thread per destination index d: the float32 tap position, cv2's interpolateCubic with A = -0.75 and the weights
// rounded to 1/2048.  Every operation is an explicit _rn intrinsic so that no FMA contraction changes a weight.
__global__ void __launch_bounds__(256)
resize_cubic_table_kernel(int n_src, int n_dst, double scale, int4 *__restrict__ idx, short4 *__restrict__ w)
{
    const int d = blockIdx.x * blockDim.x + threadIdx.x;
    if (d >= n_dst) return;
    float f = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn((double)d, 0.5), scale), -0.5));
    const float fl = floorf(f);
    const int s = (int)fl;
    f = __fsub_rn(f, fl);
    const float A = -0.75f;
    const float x1 = __fadd_rn(f, 1.f), g = __fsub_rn(1.f, f);
    const float c0 = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, x1), 5.f * A), x1), 8.f * A), x1), 4.f * A);
    const float c1 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, f), A + 3.f), f), f), 1.f);
    const float c2 = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.f, g), A + 3.f), g), g), 1.f);
    const float c3 = __fsub_rn(__fsub_rn(__fsub_rn(1.f, c0), c1), c2);
    auto q = [](float c) { return (short)max(-32768, min(32767, __float2int_rn(__fmul_rn(c, 2048.f)))); };
    auto tap = [&](int k) { return max(0, min(n_src - 1, s + k)); };
    idx[d] = make_int4(tap(-1), tap(0), tap(1), tap(2));
    w[d] = make_short4(q(c0), q(c1), q(c2), q(c3));
}

constexpr int kMaxRates = ORP_RESIZE_MAX_RATES;

// per rate: scaled size, offsets into the concatenated tables; rate exactly 1 has no table and is a plain crop
struct RateSet {
    int n;
    int wr[kMaxRates], hr[kMaxRates], xoff[kMaxRates], yoff[kMaxRates], identity[kMaxRates];
};

// one thread = one output pixel (all C channels) of tile blockIdx.z.  tiles[t] = (rate index, left, up) in the scaled
// image; NULL means one tile at (0, 0) of rate 0 (the full-image entry).  Pixels outside the scaled image are zero.
// The 16 taps of neighbouring threads overlap and come from L1 / L2; the table entries of a row are shared by the block.
template <int C>
__global__ void __launch_bounds__(256)
resize_tiles_cubic_kernel(const uint8_t *__restrict__ img, int W, RateSet rs, const int4 *__restrict__ xidx,
                          const short4 *__restrict__ xw, const int4 *__restrict__ yidx, const short4 *__restrict__ yw,
                          const int32_t *__restrict__ tiles, int tile_h, int tile_w, uint8_t *__restrict__ out)
{
    const int t = blockIdx.z;
    const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y * blockDim.y + threadIdx.y;
    if (x >= tile_w || y >= tile_h) return;
    int r = 0, left = 0, up = 0;
    if (tiles) r = __ldg(tiles + 3 * t), left = __ldg(tiles + 3 * t + 1), up = __ldg(tiles + 3 * t + 2);
    const long long X = (long long)left + x, Y = (long long)up + y;
    int v[C];
#pragma unroll
    for (int c = 0; c < C; ++c) v[c] = 0;
    if (r >= 0 && r < rs.n && X >= 0 && Y >= 0 && X < rs.wr[r] && Y < rs.hr[r]) {
        if (rs.identity[r]) {
            const uint8_t *p = img + ((size_t)Y * W + X) * C;
#pragma unroll
            for (int c = 0; c < C; ++c) v[c] = __ldg(p + c);
        } else {
            const int4 xi = __ldg(xidx + rs.xoff[r] + X), yi = __ldg(yidx + rs.yoff[r] + Y);
            const short4 wx = __ldg(xw + rs.xoff[r] + X), wy = __ldg(yw + rs.yoff[r] + Y);
            const int cols[4] = {xi.x, xi.y, xi.z, xi.w}, rows[4] = {yi.x, yi.y, yi.z, yi.w};
            const int wxs[4] = {wx.x, wx.y, wx.z, wx.w}, wys[4] = {wy.x, wy.y, wy.z, wy.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const uint8_t *row = img + (size_t)rows[k] * W * C;
                int h[C];
#pragma unroll
                for (int c = 0; c < C; ++c) h[c] = 0;
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    const uint8_t *p = row + (size_t)cols[j] * C;
#pragma unroll
                    for (int c = 0; c < C; ++c) h[c] += wxs[j] * (int)__ldg(p + c);
                }
#pragma unroll
                for (int c = 0; c < C; ++c) v[c] += wys[k] * h[c];
            }
#pragma unroll
            for (int c = 0; c < C; ++c) v[c] = max(0, min(255, (v[c] + (1 << 21)) >> 22));
        }
    }
    uint8_t *dst = out + (((size_t)t * tile_h + y) * tile_w + x) * C;
#pragma unroll
    for (int c = 0; c < C; ++c) dst[c] = (uint8_t)v[c];
}

// cv2's dsize = saturate_cast<int>(n * rate): round half to even (the default rounding mode of llrint); 0 if empty or bad
int dst_size(int n, double rate)
{
    if (!(rate > 0) || !isfinite(rate) || n < 1) return 0;
    const double v = (double)n * rate;
    if (!(v < 2147483647.0)) return 0;
    const long long m = llrint(v);
    return m >= 1 ? (int)m : 0;
}

int launch_resize(const uint8_t *img, int W, int C, const RateSet &rs, const int32_t *xidx, const int16_t *xw,
                  const int32_t *yidx, const int16_t *yw, const int32_t *tiles, int ntiles, int tile_h, int tile_w,
                  uint8_t *out, cudaStream_t st)
{
    const dim3 block(128, 2);
    const dim3 grid((tile_w + 127) / 128, (tile_h + 1) / 2, ntiles);
    const int4 *xi = reinterpret_cast<const int4 *>(xidx), *yi = reinterpret_cast<const int4 *>(yidx);
    const short4 *xs = reinterpret_cast<const short4 *>(xw), *ys = reinterpret_cast<const short4 *>(yw);
    switch (C) {
    case 1: resize_tiles_cubic_kernel<1><<<grid, block, 0, st>>>(img, W, rs, xi, xs, yi, ys, tiles, tile_h, tile_w, out); break;
    case 2: resize_tiles_cubic_kernel<2><<<grid, block, 0, st>>>(img, W, rs, xi, xs, yi, ys, tiles, tile_h, tile_w, out); break;
    case 3: resize_tiles_cubic_kernel<3><<<grid, block, 0, st>>>(img, W, rs, xi, xs, yi, ys, tiles, tile_h, tile_w, out); break;
    default: resize_tiles_cubic_kernel<4><<<grid, block, 0, st>>>(img, W, rs, xi, xs, yi, ys, tiles, tile_h, tile_w, out); break;
    }
    ORP_LAUNCHED();
    return ORP_OK;
}

bool misaligned(const void *p, size_t a) { return reinterpret_cast<uintptr_t>(p) % a != 0; }

// tables of the non-identity rates present and aligned (idx int4, weights short4)
bool bad_tables(const RateSet &rs, const int32_t *xidx, const int16_t *xw, const int32_t *yidx, const int16_t *yw)
{
    bool need = false;
    for (int r = 0; r < rs.n; ++r) need |= !rs.identity[r];
    if (!need) return false;
    return !xidx || !xw || !yidx || !yw || misaligned(xidx, 16) || misaligned(yidx, 16) || misaligned(xw, 8) ||
           misaligned(yw, 8);
}

}  // namespace
}  // namespace orp

extern "C" int orp_resize_cubic_table(int n_src, double rate, int n_dst, int32_t *idx, int16_t *w, void *stream)
{
    using namespace orp;
    if (!idx || !w || misaligned(idx, 16) || misaligned(w, 8))
        return fail(ORP_EINVAL, "orp_resize_cubic_table: idx (16-byte aligned) and w (8-byte aligned) are required");
    if (n_src < 1 || dst_size(n_src, rate) < 1 || n_dst != dst_size(n_src, rate))
        return fail(ORP_EINVAL, "orp_resize_cubic_table: rate must be > 0 and n_dst = round_half_even(n_src * rate) >= 1");
    int rc = ensure_device();
    if (rc) return rc;
    resize_cubic_table_kernel<<<(n_dst + 255) / 256, 256, 0, static_cast<cudaStream_t>(stream)>>>(
        n_src, n_dst, 1.0 / rate, reinterpret_cast<int4 *>(idx), reinterpret_cast<short4 *>(w));
    ORP_LAUNCHED();
    return ORP_OK;
}

extern "C" int orp_resize_tiles_cubic_u8(const uint8_t *img_hwc, int H, int W, int C, int nrates, const double *rates,
                                         const int32_t *xidx, const int16_t *xw, const int32_t *yidx, const int16_t *yw,
                                         const int32_t *tiles, int ntiles, int subsize, uint8_t *out, void *stream)
{
    using namespace orp;
    if (!img_hwc || !tiles || !out || !rates || H < 1 || W < 1 || C < 1 || C > 4 || ntiles < 0 || ntiles > 65535 ||
        subsize < 1 || nrates < 1 || nrates > kMaxRates)
        return fail(ORP_EINVAL, "orp_resize_tiles_cubic_u8: bad arguments (1 <= C <= 4, 0 <= ntiles <= 65535, "
                                "1 <= nrates <= ORP_RESIZE_MAX_RATES)");
    RateSet rs{};
    rs.n = nrates;
    int xoff = 0, yoff = 0;
    for (int r = 0; r < nrates; ++r) {
        rs.wr[r] = dst_size(W, rates[r]);
        rs.hr[r] = dst_size(H, rates[r]);
        if (rs.wr[r] < 1 || rs.hr[r] < 1)
            return fail(ORP_EINVAL, "orp_resize_tiles_cubic_u8: every rate must be > 0 and give a non-empty image");
        rs.identity[r] = rates[r] == 1.0;
        rs.xoff[r] = xoff;
        rs.yoff[r] = yoff;
        if (!rs.identity[r]) {
            if (xoff > INT32_MAX - rs.wr[r] || yoff > INT32_MAX - rs.hr[r])
                return fail(ORP_EINVAL, "orp_resize_tiles_cubic_u8: tables too large");
            xoff += rs.wr[r];
            yoff += rs.hr[r];
        }
    }
    if (bad_tables(rs, xidx, xw, yidx, yw))
        return fail(ORP_EINVAL, "orp_resize_tiles_cubic_u8: the tables of every rate != 1 are required (aligned)");
    int rc = ensure_device();
    if (rc) return rc;
    if (ntiles == 0) return ORP_OK;
    return launch_resize(img_hwc, W, C, rs, xidx, xw, yidx, yw, tiles, ntiles, subsize, subsize, out,
                         static_cast<cudaStream_t>(stream));
}

extern "C" int orp_resize_cubic_u8(const uint8_t *img_hwc, int H, int W, int C, double rate, const int32_t *xidx,
                                   const int16_t *xw, const int32_t *yidx, const int16_t *yw, uint8_t *out, void *stream)
{
    using namespace orp;
    RateSet rs{};
    rs.n = 1;
    rs.wr[0] = dst_size(W, rate);
    rs.hr[0] = dst_size(H, rate);
    rs.identity[0] = rate == 1.0;
    if (!img_hwc || !out || H < 1 || W < 1 || C < 1 || C > 4 || rs.wr[0] < 1 || rs.hr[0] < 1 || rs.hr[0] > 131070)
        return fail(ORP_EINVAL, "orp_resize_cubic_u8: bad arguments (1 <= C <= 4, rate > 0, non-empty result)");
    if (bad_tables(rs, xidx, xw, yidx, yw))
        return fail(ORP_EINVAL, "orp_resize_cubic_u8: the tables are required (aligned) unless rate == 1");
    int rc = ensure_device();
    if (rc) return rc;
    return launch_resize(img_hwc, W, C, rs, xidx, xw, yidx, yw, nullptr, 1, rs.hr[0], rs.wr[0], out,
                         static_cast<cudaStream_t>(stream));
}

extern "C" int orp_split_tiles_u8(const uint8_t *img_hwc, int H, int W, int C, const int32_t *origins, int ntiles, int subsize,
                                  uint8_t *out, void *stream)
{
    using namespace orp;
    if (!img_hwc || !origins || !out || H < 1 || W < 1 || C < 1 || ntiles < 0 || subsize < 1 || ((size_t)subsize * C) % 4)
        return fail(ORP_EINVAL, "orp_split_tiles_u8: bad arguments (subsize*C must be a multiple of 4)");
    int rc = ensure_device();
    if (rc) return rc;
    if (ntiles == 0) return ORP_OK;
    const size_t total = (size_t)ntiles * subsize * ((size_t)subsize * C / 4);
    split_tiles_kernel<<<grid_for(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(img_hwc, H, W, C, origins, ntiles,
                                                                                           subsize, out);
    ORP_LAUNCHED();
    return ORP_OK;
}
