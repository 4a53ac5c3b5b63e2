// Compiles the LOAM front-end adaptor (b200host::FeatureExtraction, the device-cloud overloads of ScanToMap::scan2MapOptimization
// and KeyframeStore::add) against the C ABI and runs the full chain raw scan -> features -> optimize -> store -> local map (used by
// tests/test_gpu_loam_features.py).  Without a GPU it fails loudly when the first handle is created.
#include <cmath>
#include <cstdio>
#include <cstdint>

#include "ndt_gpu.hpp"
#include "scan2map_gpu.hpp"

struct PointXYZIR {  // layout of velodyne_ros::Point without the time field: x y z (pad) intensity ring
    float x, y, z, pad, intensity;
    uint16_t ring;
    uint16_t pad1;
    float pad2, pad3;
};
struct Cloud { std::vector<float> points; };

// a 16-ring spin inside a 40 m x 24 m box room with a pillar, 1800 azimuths
static std::vector<PointXYZIR> room_scan(float ox) {
    std::vector<PointXYZIR> pts;
    for (int c = 0; c < 1800; ++c) {
        const double az = 2 * M_PI * c / 1800;
        for (int r = 0; r < 16; ++r) {
            const double el = (-15.0 + 2.0 * r) * M_PI / 180.0;
            const double dx = std::cos(el) * std::cos(az), dy = std::cos(el) * std::sin(az), dz = std::sin(el);
            double t = 1e9;
            if (dx > 0) t = std::fmin(t, (20.0 - ox) / dx);
            if (dx < 0) t = std::fmin(t, (-20.0 - ox) / dx);
            if (dy > 0) t = std::fmin(t, 12.0 / dy);
            if (dy < 0) t = std::fmin(t, -12.0 / dy);
            if (dz < 0) t = std::fmin(t, -1.5 / dz);
            if (dz > 0) t = std::fmin(t, 4.0 / dz);
            if (std::fabs(az - 0.5) < 0.08) t = std::fmin(t, 6.0);  // pillar
            PointXYZIR p{};
            p.x = (float)(t * dx); p.y = (float)(t * dy); p.z = (float)(t * dz);
            p.intensity = (float)(c % 50);
            p.ring = (uint16_t)r;
            pts.push_back(p);
        }
    }
    return pts;
}

int main() {
    using namespace b200host;
    try {
        b200_feature_params fp{16, 1800, 1, 0, 1.0f, 1000.0f, 1.0f, 0.1f, 0.4f, 0.2f, 0.4f, 0};
        FeatureExtraction<PointXYZIR> fe(fp);
        KeyframeStore<Cloud> store;
        ScanToMap<Cloud> s2m(400000);
        b200_surround_params sp{50.f, 2.f, 0.2f, 0.4f};
        float t6[6] = {0, 0, 0, 0, 0, 0};
        for (int k = 0; k < 5; ++k) {
            if (!fe.extract(room_scan(0.5f * k))) return 3;
            int64_t nc = 0, ns = 0;
            const void* c = fe.deviceCloud(B200_FEATURES_CORNER_DS, &nc);
            const void* s = fe.deviceCloud(B200_FEATURES_SURF_DS, &ns);
            if (k > 0) {
                if (!s2m.extractSurroundingKeyFrames(store, -1, (double)k, sp)) return 4;
                s2m.scan2MapOptimization(c, nc, s, ns, t6);
            }
            const float pose[6] = {0.5f * k, 0.f, 0.f, 0.f, 0.f, 0.f};
            if (store.add(c, nc, s, ns, pose, (double)k) != k) return 5;
            std::printf("scan %d: extracted %lld corner %lld surf %lld ds %lld / %lld t6 x %.4f\n", k, (long long)fe.info().n_extracted,
                        (long long)fe.info().n_corner, (long long)fe.info().n_surface, (long long)nc, (long long)ns, t6[3]);
            if (nc < 1 || ns < 100) return 6;
        }
        if (store.size() != 5 || !std::isfinite(t6[3])) return 7;
    } catch (const std::exception& e) {
        std::printf("FAILED LOUDLY: %s\n", e.what());
        return 10;
    }
    std::printf("features chain ok\n");
    return 0;
}
