// beam_emul.cpp -- TEST-ONLY host compilation of the per-pixel candidate lists of rt_device.cuh (pixel_beam,
// pixel_candidates) next to emul.cpp's entry points, for tests/test_camera_lists.py.  Never part of the product.
#include "emul.cpp"

extern "C" {
// For camera ray i = (pixel pix[i], jitter (u[2i], u[2i+1]) in [0, 1)) of the scene's camera: out[4i..4i+3] =
//   list length of the pixel (kPixelTraverse when its rays take the index traversal),
//   leaves the index traversal of the ray reaches (as collect_leaf_hits walks it) that are NOT in the list,
//   id from the list (closest plane, leaf_test of each candidate, replay_reference; -2 for a traverse pixel),
//   id from scene_intersect<0> (collect_leaf_hits + replay_reference) before the final distance is recomputed.
void emu_camera_lists(void* h, long n, const uint32_t* pix, const float* u, int32_t* out) {
    const DevScene& S = ((EmuScene*)h)->dev;
#pragma omp parallel for schedule(dynamic, 64)
    for (long i = 0; i < n; ++i) {
        const uint32_t pixel = pix[i], x = pixel % S.width, y = pixel / S.width;
        float fx = __fadd_rn((float)x, u[2 * i]), fy = __fadd_rn((float)y, u[2 * i + 1]);   // camera_path's jitter
        if (S.dialect == DIALECT_HW3) { fx = __fadd_rn(fx, 0.5f); fy = __fadd_rn(fy, 0.5f); }
        vec3 o, d;
        camera_ray(S.cam, S.width, S.height, fx, fy, o, d);
        const Beam B = pixel_beam(S.cam, S.width, S.height, S.dialect, x, y);
        uint32_t list[kMaxRecords];
        const uint32_t len = pixel_candidates(S, B, list, nullptr);
        // the leaves the ray's own traversal reaches: collect_leaf_hits' walk, every leaf it would leaf_test
        int missing = 0;
        if (S.iroot != IREF_NONE) {
            const vec3 inv = ray_inv(d), oi = o * inv;
            const ConeDir dn = cone_dir(d);
            std::vector<uint32_t> st{S.iroot};
            while (!st.empty()) {
                const uint32_t ref = st.back();
                st.pop_back();
                if (ref & IREF_LEAF) {
                    if (len != kPixelTraverse && std::find(list, list + len, ref) == list + len) ++missing;
                    continue;
                }
                NodeVisit v = index_visit(S, ref, inv, oi, dn);
                for (int c = 0; c < (int)kNodeWidth; ++c)
                    if (v.hit[c]) st.push_back(v.ref[c]);
            }
        }
        float cd; int pid;
        closest_plane(S, o, d, cd, pid);
        int id_list = -2;
        if (len != kPixelTraverse) {
            const vec3 inv = ray_inv(d), oi = o * inv;
            LeafRec rec[kMaxRecords];
            int k = 0;
            for (uint32_t j = 0; j < len; ++j) {
                float bt, tc; int bid;
                if (leaf_test(S, list[j], o, d, inv, oi, bt, bid, tc, nullptr) && bid >= 0) {
                    rec[k].key = list[j] & 0xFFFFFFu; rec[k].id = bid; rec[k].t = bt; rec[k].tcull = tc;
                    ++k;
                }
            }
            const BestHit b = replay_reference(S, o, d, cd, rec, k);
            id_list = (b.id != -1 && b.t < cd) ? b.id : pid;
        }
        const SceneHit ht = scene_intersect<0>(S, o, d, nullptr, nullptr, nullptr);
        out[4 * i] = (int32_t)len;
        out[4 * i + 1] = missing;
        out[4 * i + 2] = id_list;
        out[4 * i + 3] = ht.id;
    }
}
// The list length of every pixel of the scene's camera (kPixelTraverse: index traversal)
void emu_camera_list_lengths(void* h, uint32_t* out) {
    const DevScene& S = ((EmuScene*)h)->dev;
    const long npix = (long)S.width * S.height;
#pragma omp parallel for schedule(dynamic, 64)
    for (long p = 0; p < npix; ++p) {
        uint32_t list[kMaxRecords];
        out[p] = pixel_candidates(S, pixel_beam(S.cam, S.width, S.height, S.dialect, (uint32_t)(p % S.width), (uint32_t)(p / S.width)),
                                  list, nullptr);
    }
}
}
