// render_shim.cpp -- TEST INFRASTRUCTURE ONLY.  dfb_render (dynamicfusion_body_b200/csrc/render.cu) as a serial loop over HOST
// pointers, around the very same per-face and per-pixel functions (csrc/dfb_render.h), so that the CPU test-suite can check the
// rasteriser against the oracle (oracle/render.py) on a box that has no GPU.  The z-buffer min is order-independent, so the
// serial loop computes what the device's atomics do.  Build with -ffp-contract=off.  The product never loads this library.
#include "../../include/dfb.h"
#include "../../dynamicfusion_body_b200/csrc/dfb_render.h"

using namespace dfb;

extern "C" int rs_render(const double* pts, int64_t n_pts, const int32_t* faces, int64_t n_faces, const dfb_views* views,
                         uint64_t* zbuf, float* depth, int32_t* face, float* normal) {
    const int V = views->n_views, rows = views->rows, cols = views->cols;
    const int64_t npix = (int64_t)rows * cols;
    for (int64_t p = 0; p < V * npix; ++p) zbuf[p] = DFB_RENDER_EMPTY;
    for (int v = 0; v < V; ++v) {
        uint64_t* zv = zbuf + v * npix;
        for (int64_t t = 0; t < n_faces; ++t) {
            RenderFace f;
            if (!render_face_setup(pts, n_pts, faces, t, views->K, views->has_extrinsics ? views->E[v] : nullptr, rows, cols, &f)) continue;
            for (int r = f.r0; r <= f.r1; ++r)
                for (int c = f.c0; c <= f.c1; ++c) {
                    uint64_t key;
                    if (render_pixel_key(f, r, c, (uint32_t)t, &key) && key < zv[(int64_t)r * cols + c]) zv[(int64_t)r * cols + c] = key;
                }
        }
    }
    for (int64_t p = 0; p < V * npix; ++p) render_resolve(zbuf[p], pts, faces, depth + p, face + p, normal + 3 * p);
    return DFB_OK;
}
