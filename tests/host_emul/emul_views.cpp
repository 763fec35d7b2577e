// emul_views.cpp -- TEST-ONLY: the host emulation of emul.cpp plus the host side of rtc_scene_set_camera, for
// tests/test_views.py.  Like emul.cpp, never part of librtc_b200.so.
#include "emul.cpp"

extern "C" {
// The camera (13 floats: position, right, up, forward, fov_x), and the index BVH rebuilt for it when it lies beyond the
// extent the tree was built for, as c_api.cu ensure_index_extent does.  Returns 1 when the tree was rebuilt.
int emu_set_camera(void* h, const float* c) {
    EmuScene* e = (EmuScene*)h;
    Camera& cam = e->host.cam;
    cam.pos = mk3(c[0], c[1], c[2]); cam.right = mk3(c[3], c[4], c[5]); cam.up = mk3(c[6], c[7], c[8]);
    cam.forward = mk3(c[9], c[10], c[11]); cam.fov_x = c[12];
    const double extent = std::max({std::fabs((double)c[0]), std::fabs((double)c[1]), std::fabs((double)c[2])});
    const bool rebuild = extent > e->host.flat.index_extent;
    if (rebuild) e->host.build_index(extent);
    // build_index replaces the index nodes and the unit boxes; every scalar (the camera among them) follows the host scene
    e->dev.inodes = (const float4*)e->host.flat.inodes.data();
    e->dev.ubox = (const float4*)e->host.flat.ubox.data();
    fill_dev_scalars(e->host, e->dev);
    return rebuild ? 1 : 0;
}
}
