// Compiles the scan-to-map local map adaptor (b200host::KeyframeStore::add + ScanToMap::extractSurroundingKeyFrames) against the
// C ABI and runs it (used by tests/test_loam_local_map_cpu.py and tests/test_gpu_loam_local_map.py).  Without a GPU it must
// fail loudly when the store is created; with one it stores 30 keyframes of a walled room along a line and builds the local
// map of the last one.
#include <cmath>
#include <cstdio>
#include <random>

#include "ndt_gpu.hpp"
#include "scan2map_gpu.hpp"

struct PointXYZI {  // layout of pcl::PointXYZI: 32 bytes
    float x, y, z, pad, intensity, pad1, pad2, pad3;
};
struct Cloud { std::vector<PointXYZI> points; };

int main() {
    using namespace b200host;
    std::mt19937 rng(5);
    std::uniform_real_distribution<float> u(-20.f, 20.f), h(0.f, 4.f);
    try {
        KeyframeStore<Cloud> store;
        const int K = 30;
        for (int k = 0; k < K; ++k) {
            Cloud corner, surf;
            for (int i = 0; i < 400; ++i) {
                PointXYZI p{};
                p.x = u(rng); p.y = 10.f; p.z = h(rng);   // a wall 10 m to the left, in the lidar frame
                (i % 4 == 0 ? corner : surf).points.push_back(p);
            }
            const float pose[6] = {(float)k, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (store.add(corner, surf, pose, (double)k) != k) return 3;
        }
        ScanToMap<Cloud> s2m(200000);
        b200_surround_params prm{50.f, 2.f, 0.2f, 0.4f};
        if (!s2m.extractSurroundingKeyFrames(store, -1, (double)K, prm)) return 4;
        const b200_surround_info& in = s2m.surroundInfo();
        std::printf("list %lld kept %lld raw %lld / %lld ds %lld / %lld\n", (long long)in.n_list, (long long)in.n_kept, (long long)in.n_corner_raw,
                    (long long)in.n_surf_raw, (long long)in.n_corner, (long long)in.n_surf);
        // 30 keyframes 1 m apart: 15 key-pose leaves of 2 m, then the 9 keyframes of the last 10 s
        if (in.n_list != 15 + 9 || in.n_kept != in.n_list || in.n_corner_raw != 100 * in.n_kept || in.n_corner < 1 || in.n_surf < 1) return 5;
    } catch (const std::exception& e) {
        std::printf("FAILED LOUDLY: %s\n", e.what());
        return 10;
    }
    std::printf("local map adaptor ok\n");
    return 0;
}
