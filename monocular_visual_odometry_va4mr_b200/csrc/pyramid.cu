// Image pyramid construction for the pyramidal LK tracker (replaces OpenCV's
// buildOpticalFlowPyramid / pyrDown behind cv2.calcOpticalFlowPyrLK, reference
// VisualOdometryPipeLine.py:281,287; spec SURVEY.md A.1).
//
// HBM layout: one "slab" per frame holding every level with a materialised REFLECT_101
// border of VO_BORDER pixels on all four sides (cv2 does the same with copyMakeBorder), so
// that the tracker's window reads and the 5x5 / 3x3 stencils never branch on the image edge.
// Row pitch is a multiple of 128 B and pixel (0,0) of every level is 32 B aligned.
#include "internal.cuh"
#include "tma.cuh"

int vo_pyr_levels(int w, int h, int win_w, int win_h, int max_level)
{
    int levels = 1;
    for (int l = 1; l <= max_level && levels < VO_MAX_LEVELS; ++l) {
        w = (w + 1) / 2;
        h = (h + 1) / 2;
        if (w <= win_w || h <= win_h) break;
        ++levels;
    }
    return levels;
}

void vo_pyr_geom(int rows, int cols, int levels, PyrGeom* g)
{
    g->levels = levels;
    size_t off = 256;  // front pad: word-aligned staging may touch a few bytes before row -VO_BORDER
    int w = cols, h = rows;
    for (int l = 0; l < levels; ++l) {
        g->w[l] = w;
        g->h[l] = h;
        g->pitch[l] = (int)vo_align((size_t)w + 2 * VO_BORDER, 128);
        off = vo_align(off, 256);
        g->off[l] = off + (size_t)VO_BORDER * g->pitch[l] + VO_BORDER;
        off += (size_t)g->pitch[l] * (h + 2 * VO_BORDER);
        w = (w + 1) / 2;
        h = (h + 1) / 2;
    }
    g->slab_bytes = vo_align(off, 256) + 256;
}

void vo_seq_ext(int rows, int cols, int win_w, int win_h, int max_level, VoSeqExt* e)
{
    *e = VoSeqExt{};
    e->levels = vo_pyr_levels(cols, rows, win_w, win_h, max_level);
    for (int l = 0; l < e->levels; ++l) {
        e->w[l] = cols; e->h[l] = rows;
        cols = (cols + 1) / 2; rows = (rows + 1) / 2;
    }
}

Pyramid vo_pyramid_at(const PyrGeom& g, uint8_t* slab)
{
    Pyramid p;
    p.levels = g.levels;
    for (int l = 0; l < g.levels; ++l) {
        p.lv[l].base = slab + g.off[l];
        p.lv[l].w = g.w[l];
        p.lv[l].h = g.h[l];
        p.lv[l].pitch = g.pitch[l];
    }
    return p;
}

__device__ __forceinline__ int reflect101(int p, int len)
{
    // general (multi-bounce) REFLECT_101; len >= 2
    while (p < 0 || p >= len) p = p < 0 ? -p : 2 * len - 2 - p;
    return p;
}

// raw image (rows of raw_row bytes) -> bordered level 0.  One thread = one 16-byte store of the bordered row.
// ext: the sequence's own width and height (the grid covers the slot's); list: raw image z goes to slab list[z]
__global__ void __launch_bounds__(256)
pad_level0_kernel(const uint8_t* __restrict__ raw, size_t raw_stride, size_t raw_row, int w, int h,
                  uint8_t* __restrict__ slab, size_t slab_stride, size_t off0, int pitch, const VoSeqExt* __restrict__ ext,
                  const int* __restrict__ list)
{
    const int seq = list ? list[blockIdx.z] : blockIdx.z;
    if (ext) { w = ext[seq].w[0]; h = ext[seq].h[0]; }
    const uint8_t* src = raw + blockIdx.z * raw_stride;
    uint8_t* dst = slab + seq * slab_stride + off0;
    const int gx = (blockIdx.x * blockDim.x + threadIdx.x) * 16 - VO_BORDER;  // first of 16 px
    const int gy = blockIdx.y * blockDim.y + threadIdx.y - VO_BORDER;
    if (gx >= w + VO_BORDER || gy >= h + VO_BORDER) return;
    const int sy = reflect101(gy, h);
    const uint8_t* srow = src + (size_t)sy * raw_row;
    uint32_t v[4];
    if (gx >= 0 && gx + 15 < w) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const uint8_t* s = srow + gx + 4 * k;
            v[k] = (uint32_t)__ldg(s) | ((uint32_t)__ldg(s + 1) << 8) | ((uint32_t)__ldg(s + 2) << 16) |
                   ((uint32_t)__ldg(s + 3) << 24);
        }
    } else {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            uint32_t acc = 0;
#pragma unroll
            for (int b = 0; b < 4; ++b) {
                int x = gx + 4 * k + b;
                uint32_t px = (x < w + VO_BORDER) ? __ldg(srow + reflect101(x, w)) : 0u;
                acc |= px << (8 * b);
            }
            v[k] = acc;
        }
    }
    // pitch >= w + 2*VO_BORDER rounded up to 128, so a 16-byte store never leaves the row
    *reinterpret_cast<uint4*>(dst + (long long)gy * pitch + gx) = make_uint4(v[0], v[1], v[2], v[3]);
}

// level l (bordered) -> level l+1 (bordered).  One thread = 4 consecutive pixels of the
// bordered destination row; 5x5 binomial [1 4 6 4 1]^2, (sum+128)>>8.
__global__ void __launch_bounds__(256)
pyr_down_kernel(const uint8_t* __restrict__ slab_src, uint8_t* __restrict__ slab_dst, size_t slab_stride,
                size_t off_s, int sw, int sh, int spitch, size_t off_d, int dw, int dh, int dpitch,
                const VoSeqExt* __restrict__ ext, int level, const int* __restrict__ list)
{
    const int seq = list ? list[blockIdx.z] : blockIdx.z;
    if (ext) {   // the sequence's own level `level` from its level - 1; nothing beyond its level count
        if (level >= ext[seq].levels) return;
        dw = ext[seq].w[level]; dh = ext[seq].h[level];
    }
    const uint8_t* src = slab_src + seq * slab_stride + off_s;
    uint8_t* dst = slab_dst + seq * slab_stride + off_d;
    const int gx = (blockIdx.x * blockDim.x + threadIdx.x) * 4 - VO_BORDER;
    const int gy = blockIdx.y * blockDim.y + threadIdx.y - VO_BORDER;
    if (gx >= dw + VO_BORDER || gy >= dh + VO_BORDER) return;
    const int ry = reflect101(gy, dh);
    uint32_t out = 0;
    if (gx >= 0 && gx + 3 < dw) {
        // interior fast path: 4 outputs share an 11-byte source footprint per row
        int acc[4] = {0, 0, 0, 0};
        const int wy[5] = {1, 4, 6, 4, 1};
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            const uint8_t* s = src + (long long)(2 * ry - 2 + r) * spitch + (2 * gx - 2);
            int p[11];
#pragma unroll
            for (int k = 0; k < 11; ++k) p[k] = __ldg(s + k);
#pragma unroll
            for (int o = 0; o < 4; ++o)
                acc[o] += wy[r] * (p[2 * o] + 4 * p[2 * o + 1] + 6 * p[2 * o + 2] + 4 * p[2 * o + 3] + p[2 * o + 4]);
        }
#pragma unroll
        for (int o = 0; o < 4; ++o) out |= (uint32_t)((acc[o] + 128) >> 8) << (8 * o);
    } else {
#pragma unroll
        for (int o = 0; o < 4; ++o) {
            int x = gx + o;
            if (x >= dw + VO_BORDER) break;
            int rx = reflect101(x, dw);
            int acc = 0;
            const int wy[5] = {1, 4, 6, 4, 1};
#pragma unroll
            for (int r = 0; r < 5; ++r) {
                const uint8_t* s = src + (long long)(2 * ry - 2 + r) * spitch + (2 * rx - 2);
                acc += wy[r] * (__ldg(s) + 4 * __ldg(s + 1) + 6 * __ldg(s + 2) + 4 * __ldg(s + 3) + __ldg(s + 4));
            }
            out |= (uint32_t)((acc + 128) >> 8) << (8 * o);
        }
    }
    *reinterpret_cast<uint32_t*>(dst + (long long)gy * dpitch + gx) = out;
}

// ---- TMA path: level l (bordered) -> interior of level l+1 -------------------------------------
// One CTA produces a 128 x 16 tile of the destination.  Its (2*128+4) x (2*16+4) source halo tile is
// fetched by two overlapping cp.async.bulk.tensor.3d boxes (x, y, sequence; a TMA box is at most 256
// wide) into shared memory -- the materialised
// REFLECT_101 border means no tile ever needs edge handling, and reads past the slab row are zero
// filled by the TMA unit.  Each thread then produces 4 pixels x 2 rows: 64-bit shared-memory loads,
// the horizontal [1 4 6 4] taps as one dp4a (+1 byte), rows combined with [1 4 6 4 1], 32-bit stores
// (a warp writes 128 contiguous bytes per row).
#define PD_TW 128
#define PD_TH 16
#define PD_SB 160                // staged bytes per row of one half tile (TMA box width <= 256, multiple of 16)
#define PD_SR (2 * PD_TH + 4)    // staged rows

__global__ void __launch_bounds__(256)
pyr_down_tma_kernel(const __grid_constant__ CUtensorMap src_map, uint8_t* __restrict__ slab_dst, size_t slab_stride,
                    size_t off_d, int dw, int dh, int dpitch, int fuse_border, const VoSeqExt* __restrict__ ext, int level,
                    const int* __restrict__ list)
{
    // source bytes [0,160) and [128,288) of each row; each half starts on a 128-byte boundary (TMA destination)
    __shared__ __align__(128) uint8_t tile[2][(PD_SR * PD_SB + 127) / 128 * 128];
    __shared__ __align__(8) unsigned long long bar;
    const int seq = list ? list[blockIdx.z] : blockIdx.z;   // the slab, and the map's third coordinate
    const int X0 = blockIdx.x * PD_TW, Y0 = blockIdx.y * PD_TH;
    if (ext) {   // the sequence's own extents of this level: tiles outside them (and levels beyond its count) exit
        if (level >= ext[seq].levels) return;
        dw = ext[seq].w[level]; dh = ext[seq].h[level];
        if (X0 >= dw || Y0 >= dh) return;
        fuse_border = dw >= VO_BORDER + 2 && dh >= VO_BORDER + 2;
    }
    const uint32_t bar_a = smem_u32(&bar);
    if (threadIdx.x == 0) {
        mbar_init(bar_a, 1);
        mbar_fence_init();
        mbar_expect_tx(bar_a, 2 * PD_SR * PD_SB);
        // source coordinates in the bordered frame.  The innermost box coordinate must be a multiple of
        // 16 bytes: the tile starts 14 pixels left of the first tap (x = 2*X0 - 2 + border - 14 = 2*X0 + 16).
        tma_load_3d(smem_u32(tile[0]), &src_map, 2 * X0 + 16, 2 * Y0 - 2 + VO_BORDER, seq, bar_a);
        tma_load_3d(smem_u32(tile[1]), &src_map, 2 * X0 + 16 + 128, 2 * Y0 - 2 + VO_BORDER, seq, bar_a);
    }
    __syncthreads();
    mbar_wait(bar_a, 0);
    uint8_t* dst = slab_dst + seq * slab_stride + off_d;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
    const int x = X0 + 4 * tx;
    if (x >= dw) return;
#pragma unroll
    for (int rr = 0; rr < 2; ++rr) {
        const int yl = ty + 8 * rr;
        const int y = Y0 + yl;
        if (y >= dh) continue;
        int acc[4] = {0, 0, 0, 0};
#pragma unroll
        for (int r = 0; r < 5; ++r) {
            // taps of output pixel o start at tile byte 8*tx + 14 + 2*o; bytes 8*tx+8 .. 8*tx+27 are loaded
            const uint8_t* rowb = tile[tx >> 4] + (2 * yl + r) * PD_SB + 8 * (tx & 15) + 8;
            const uint2 lo = *reinterpret_cast<const uint2*>(rowb), hi = *reinterpret_cast<const uint2*>(rowb + 8);
            const uint32_t w1 = lo.y, w2 = hi.x, w3 = hi.y, w4 = *reinterpret_cast<const uint32_t*>(rowb + 16);
            const int wy = (r == 0 || r == 4) ? 1 : (r == 2 ? 6 : 4);
            const uint32_t q0 = __funnelshift_r(w1, w2, 16), q2 = __funnelshift_r(w2, w3, 16);
            const int h0 = __dp4a(q0, 0x04060401u, (w2 >> 16) & 0xffu);
            const int h1 = __dp4a(w2, 0x04060401u, w3 & 0xffu);
            const int h2 = __dp4a(q2, 0x04060401u, (w3 >> 16) & 0xffu);
            const int h3 = __dp4a(w3, 0x04060401u, w4 & 0xffu);
            acc[0] += wy * h0; acc[1] += wy * h1; acc[2] += wy * h2; acc[3] += wy * h3;
        }
        const uint32_t o0 = (uint32_t)((acc[0] + 128) >> 8), o1 = (uint32_t)((acc[1] + 128) >> 8);
        const uint32_t o2 = (uint32_t)((acc[2] + 128) >> 8), o3 = (uint32_t)((acc[3] + 128) >> 8);
        uint8_t* dp = dst + (long long)y * dpitch + x;
        const uint32_t word = o0 | (o1 << 8) | (o2 << 16) | (o3 << 24);
        if (x + 3 < dw) *reinterpret_cast<uint32_t*>(dp) = word;
        else { dp[0] = (uint8_t)o0; if (x + 1 < dw) dp[1] = (uint8_t)o1; if (x + 2 < dw) dp[2] = (uint8_t)o2; }
        // REFLECT_101 ring of this level written by the pixels it mirrors (dw, dh >= VO_BORDER + 2: single bounce):
        // columns 1..B -> -1..-B and dw-1-B..dw-2 -> dw..dw+B-1, rows likewise, corners by both
        if (fuse_border && (x <= VO_BORDER || x + 3 >= dw - 1 - VO_BORDER || y <= VO_BORDER || y >= dh - 1 - VO_BORDER)) {
            auto put_row = [&](int yy) {
                uint8_t* rowp = dst + (long long)yy * dpitch;
                if (yy != y) {
                    if (x + 3 < dw) *reinterpret_cast<uint32_t*>(rowp + x) = word;
                    else { rowp[x] = (uint8_t)o0; if (x + 1 < dw) rowp[x + 1] = (uint8_t)o1; if (x + 2 < dw) rowp[x + 2] = (uint8_t)o2; }
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    const int c = x + k;
                    if (c < dw) {
                        const uint8_t px = (uint8_t)(word >> (8 * k));
                        if (c >= 1 && c <= VO_BORDER) rowp[-c] = px;
                        if (c >= dw - 1 - VO_BORDER && c <= dw - 2) rowp[2 * (dw - 1) - c] = px;
                    }
                }
            };
            put_row(y);
            if (y >= 1 && y <= VO_BORDER) put_row(-y);
            if (y >= dh - 1 - VO_BORDER && y <= dh - 2) put_row(2 * (dh - 1) - y);
        }
    }
}

// REFLECT_101 border ring of one level from its own interior (the next level's halo tiles and the
// tracker's window reads depend on it)
struct BorderArgs { int levels; int w[VO_MAX_LEVELS], h[VO_MAX_LEVELS], pitch[VO_MAX_LEVELS]; unsigned long long off[VO_MAX_LEVELS]; };
__global__ void __launch_bounds__(256)
pyr_border_level_kernel(uint8_t* __restrict__ slab, size_t slab_stride, BorderArgs a, int level, const VoSeqExt* __restrict__ ext,
                        const int* __restrict__ list)
{
    int w = a.w[level], h = a.h[level];
    const int pitch = a.pitch[level];
    const int seq = list ? list[blockIdx.z] : blockIdx.z;
    if (ext) {   // only the sequences whose level was not given its ring by the tiles
        const VoSeqExt& e = ext[seq];
        if (level >= e.levels) return;
        w = e.w[level]; h = e.h[level];
        if (w >= VO_BORDER + 2 && h >= VO_BORDER + 2) return;
    }
    uint8_t* base = slab + seq * slab_stride + a.off[level];
    // ring in aligned 4-byte words: top + bottom bands over the full bordered width, then per interior
    // row 8 words on the left (x = -32..-1) and 9 on the right (from x = w & ~3, covering w .. w+31)
    const int wq = (w + 2 * VO_BORDER + 3) / 4;
    const int n_tb = 2 * VO_BORDER * wq;
    const int n_lr = h * 17;
    const int xa = w & ~3;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n_tb + n_lr; i += gridDim.x * blockDim.x) {
        int gx, gy;
        if (i < n_tb) {
            const int r = i / wq;
            gy = r < VO_BORDER ? r - VO_BORDER : h + (r - VO_BORDER);
            gx = (i - r * wq) * 4 - VO_BORDER;
        } else {
            const int k = i - n_tb, r = k / 17, c = k - r * 17;
            gy = r;
            gx = c < 8 ? c * 4 - VO_BORDER : xa + (c - 8) * 4;
        }
        const uint8_t* srow = base + (long long)reflect101(gy, h) * pitch;
        uint8_t* dp = base + (long long)gy * pitch + gx;
        const bool interior_row = gy >= 0 && gy < h;
        uint32_t v = 0;
        bool full = true;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const int xx = gx + b;
            const bool inner = interior_row && xx >= 0 && xx < w;     // already holds the filtered pixel
            full = full && !inner;
            const uint32_t px = (xx < w + VO_BORDER) ? srow[reflect101(xx, w)] : 0u;
            v |= px << (8 * b);
        }
        if (full) *reinterpret_cast<uint32_t*>(dp) = v;
        else {
#pragma unroll
            for (int b = 0; b < 4; ++b) if (gx + b >= w) dp[b] = (uint8_t)(v >> (8 * b));
        }
    }
}

static int pyr_src_map(b200vo_ctx* ctx, CUtensorMap* map, uint8_t* d_slab, size_t slab_stride, int batch, const PyrGeom& g, int l)
{
    uint8_t* start = d_slab + g.off[l] - (size_t)VO_BORDER * g.pitch[l] - VO_BORDER;   // bordered row -B, col -B
    const cuuint64_t dims[3] = {(cuuint64_t)g.pitch[l], (cuuint64_t)(g.h[l] + 2 * VO_BORDER), (cuuint64_t)batch};
    const cuuint64_t strides[2] = {(cuuint64_t)g.pitch[l], (cuuint64_t)slab_stride};
    const cuuint32_t box[3] = {PD_SB, PD_SR, 1};
    return vo_encode_tiled(ctx, map, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, start, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE);
}

int vo_build_pyramids(b200vo_ctx* ctx, const uint8_t* d_raw, size_t raw_stride, int rows, int cols,
                      const PyrGeom& g, uint8_t* d_slab, size_t slab_stride, int batch, cudaStream_t stream,
                      const VoSeqExt* d_ext, const VoSeqExt* h_ext, size_t raw_row, const int* d_list, const int* h_list, int n_slab)
{
    if (!raw_row) raw_row = (size_t)cols;
    // the slabs the tensor maps span: every slab of the set when the images go to listed slabs
    const int n_map = d_list ? n_slab : batch;
    {
        dim3 block(32, 8);
        int gxn = (cols + 2 * VO_BORDER + 15) / 16;
        dim3 grid((gxn + block.x - 1) / block.x, (rows + 2 * VO_BORDER + block.y - 1) / block.y, batch);
        pad_level0_kernel<<<grid, block, 0, stream>>>(d_raw, raw_stride, raw_row, cols, rows, d_slab, slab_stride,
                                                       g.off[0], g.pitch[0], d_ext, d_list);
        ctx->launches++;
    }
    if (g.levels > 1) {
        // TMA needs 16-byte aligned strides and base: slab strides are multiples of 256, pitches of 128
        const bool tma_ok = (slab_stride % 16 == 0 || n_map == 1) && (reinterpret_cast<uintptr_t>(d_slab) % 256 == 0);
        for (int l = 1; l < g.levels; ++l) {
            bool fused = false;
            if (tma_ok) {
                CUtensorMap map;
                VO_TRY(pyr_src_map(ctx, &map, d_slab, n_map == 1 ? g.slab_bytes : slab_stride, n_map, g, l - 1));
                dim3 grid((g.w[l] + PD_TW - 1) / PD_TW, (g.h[l] + PD_TH - 1) / PD_TH, batch);
                fused = g.w[l] >= VO_BORDER + 2 && g.h[l] >= VO_BORDER + 2;   // single-bounce reflection: the tiles write the ring
                pyr_down_tma_kernel<<<grid, 256, 0, stream>>>(map, d_slab, slab_stride, g.off[l], g.w[l], g.h[l], g.pitch[l], fused ? 1 : 0,
                                                              d_ext, l, d_list);
                if (h_ext) {   // the single-bounce test per sequence: a ring is left to the border kernel if any tile set could not write it
                    fused = true;
                    for (int b = 0; b < batch; ++b) {
                        const VoSeqExt& e = h_ext[h_list ? h_list[b] : b];
                        if (l < e.levels && !(e.w[l] >= VO_BORDER + 2 && e.h[l] >= VO_BORDER + 2)) fused = false;
                    }
                }
            } else {
                dim3 block(32, 8);
                int gxn = (g.w[l] + 2 * VO_BORDER + 3) / 4;
                dim3 grid((gxn + block.x - 1) / block.x, (g.h[l] + 2 * VO_BORDER + block.y - 1) / block.y, batch);
                pyr_down_kernel<<<grid, block, 0, stream>>>(d_slab, d_slab, slab_stride, g.off[l - 1], g.w[l - 1],
                                                             g.h[l - 1], g.pitch[l - 1], g.off[l], g.w[l], g.h[l],
                                                             g.pitch[l], d_ext, l, d_list);
            }
            ctx->launches++;
            if (tma_ok && !fused) {
                // the next level's halo tiles read this level's border: fill it before descending (tiny levels: multi-bounce)
                BorderArgs ba{};
                ba.levels = l + 1;
                for (int k = 0; k <= l; ++k) { ba.w[k] = g.w[k]; ba.h[k] = g.h[k]; ba.pitch[k] = g.pitch[k]; ba.off[k] = g.off[k]; }
                // only level l needs filling now: launch with a single y-slice mapped onto level l
                ba.levels = l + 1;
                pyr_border_level_kernel<<<dim3(16, 1, batch), 256, 0, stream>>>(d_slab, slab_stride, ba, l, d_ext, d_list);
                ctx->launches++;
            }
        }
    }
    VO_CUDA(ctx, cudaGetLastError());
    return 0;
}
