// Compiles the loop-closure adaptor (b200host::KeyframeStore + NdtPairBatch::closeLoops, host/ndt_gpu.hpp) against the C ABI
// and runs it (used by tests/test_loop_cpu.py and tests/test_gpu_loop_closure.py).  Without a GPU it must fail loudly when the
// store is created; with one it drives around a small room twice, storing the second lap with a 0.15 m drift, and closes the
// loop of the last keyframe.
#include <cmath>
#include <cstdio>
#include <random>

#include "ndt_gpu.hpp"

struct PointXYZI {  // layout of pcl::PointXYZI: 32 bytes
    float x, y, z, pad, intensity, pad1, pad2, pad3;
};
struct Cloud { std::vector<PointXYZI> points; };

int main() {
    using namespace b200host;
    std::mt19937 rng(17);
    std::uniform_real_distribution<float> u(-15.f, 15.f), h(0.f, 5.f), s(-3.f, 3.f);
    std::normal_distribution<float> nz(0.f, 0.01f);
    std::vector<PointXYZI> room;
    auto add = [&](float x, float y, float z) { PointXYZI p{}; p.x = x; p.y = y; p.z = z; p.intensity = std::fabs(z) * 10.f; room.push_back(p); };
    for (int i = 0; i < 6000; ++i) { add(u(rng), u(rng), nz(rng)); add(u(rng), u(rng), 5.f + nz(rng)); }
    for (int i = 0; i < 1500; ++i) {
        add(15.f + nz(rng), u(rng), h(rng)); add(-15.f + nz(rng), u(rng), h(rng));
        add(u(rng), 15.f + nz(rng), h(rng)); add(u(rng), -15.f + nz(rng), h(rng));
        add(4.f + nz(rng), s(rng), h(rng)); add(s(rng), -6.f + nz(rng), h(rng));
    }
    try {
        KeyframeStore<Cloud> store;
        const int K = 40;  // two laps of 20 keyframes on a 4 m circle
        for (int k = 0; k < K; ++k) {
            const float a = 2.f * 3.14159265f * (float)(k % 20) / 20.f, x = 4.f * std::cos(a), y = 4.f * std::sin(a);
            Cloud corner, surf;  // the room in the lidar frame (translation only), split corner / surf by index
            for (size_t i = (size_t)k; i < room.size(); i += 7) {
                PointXYZI p = room[i];
                p.x -= x; p.y -= y;
                (i % 5 == 0 ? corner : surf).points.push_back(p);
            }
            const float drift = k >= 20 ? 0.15f : 0.f;
            const float pose[6] = {x + drift, y - drift, 0.f, 0.f, 0.f, 0.f};
            if (store.add(corner, surf, pose, (double)k) != k) return 3;
        }
        b200_loop_params prm{};
        prm.search_radius = 1.0f; prm.time_gap = 10.0; prm.search_num = 2; prm.leaf = 0.2f;
        prm.min_source_points = 300; prm.min_target_points = 1000; prm.max_range = 1.7976931348623157e308;
        const std::vector<int64_t> pre = store.detect({K - 1}, prm);
        NdtPairBatch<Cloud> batch;
        batch.setResolution(1.0f);
        batch.setTransformationEpsilon(0.001);
        batch.setNeighborhoodSearchMethod(DIRECT7);
        batch.closeLoops(store, {K - 1}, {}, prm);
        const b200_loop_result& r = batch.loopResult(0);
        const float* T = batch.getFinalTransformation(0);
        std::printf("query %lld pre %lld (detect %lld) n_source %d n_target %d status %d fitness %.5f tx %.4f ty %.4f\n", (long long)r.cur,
                    (long long)r.pre, (long long)pre[0], r.n_source, r.n_target, batch.status(0), batch.getFitnessScore(0), T[12], T[13]);
        if (r.pre != pre[0] || r.pre != 19) return 4;
        // the correction undoes most of the 0.15 m drift
        if (!batch.hasConverged(0) || std::fabs(T[12] + 0.15f) > 0.1f || std::fabs(T[13] - 0.15f) > 0.1f || !(batch.getFitnessScore(0) < 0.05)) return 5;
    } catch (const std::exception& e) {
        std::printf("FAILED LOUDLY: %s\n", e.what());
        return 10;
    }
    std::printf("loop closure adaptor ok\n");
    return 0;
}
