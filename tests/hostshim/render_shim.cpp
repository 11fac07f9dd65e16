// render_shim.cpp -- TEST INFRASTRUCTURE ONLY.  dfb_render (dynamicfusion_body_b200/csrc/render.cu) as a serial loop over HOST
// pointers, around the very same set-up, per-face and per-pixel functions (csrc/dfb_render.h), so that the CPU test-suite can check
// the rasteriser against the oracle (oracle/render.py) on a box that has no GPU.  The z-buffer min is order-independent, so the
// serial loop computes what the device's atomics do.  Build with -ffp-contract=off.  The product never loads this library.
#include <vector>

#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_render.h"

using namespace dfb;

// dfb_render without its device workspace (the z-buffer is the shim's own)
extern "C" int hs_render(const double* pts, int64_t n_pts, const int32_t* faces, int64_t n_faces, const dfb_views* views, float* depth,
                         int32_t* face, float* normal) {
    RenderCams cams;
    if (int r = build_render(cams, pts, n_pts, faces, n_faces, views, depth, face, normal)) return r;
    const int64_t npix = (int64_t)cams.rows * cams.cols;
    std::vector<uint64_t> zbuf(cams.n_views * npix, DFB_RENDER_EMPTY);
    for (int v = 0; v < cams.n_views; ++v) {
        uint64_t* zv = zbuf.data() + v * npix;
        for (int64_t t = 0; t < n_faces; ++t) {
            RenderFace f;
            if (!render_face_setup(pts, n_pts, faces, t, cams.K, cams.has_e ? cams.E + 12 * v : nullptr, cams.rows, cams.cols, &f)) continue;
            for (int r = f.r0; r <= f.r1; ++r)
                for (int c = f.c0; c <= f.c1; ++c) {
                    uint64_t key;
                    if (render_pixel_key(f, r, c, (uint32_t)t, &key) && key < zv[(int64_t)r * cams.cols + c]) zv[(int64_t)r * cams.cols + c] = key;
                }
        }
    }
    for (int64_t p = 0; p < cams.n_views * npix; ++p) render_resolve(zbuf[p], pts, faces, depth + p, face + p, normal + 3 * p);
    return DFB_OK;
}
