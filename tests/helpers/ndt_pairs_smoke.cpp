// Compiles the batched loop-closure adaptor (b200host::NdtPairBatch, host/ndt_gpu.hpp) against the C ABI and runs it (used by
// tests/test_ndt_pairs_cpu.py and tests/test_gpu_ndt_pairs.py).  Without a GPU it must fail loudly at the first align(); with
// one it registers three drifted copies of a small room against the room, plus one pair with an empty source.
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
    std::mt19937 rng(11);
    std::uniform_real_distribution<float> u(-15.f, 15.f), h(0.f, 5.f), s(-3.f, 3.f);
    std::normal_distribution<float> nz(0.f, 0.01f);
    Cloud room;
    auto add = [&](Cloud& c, float x, float y, float z) { PointXYZI p{}; p.x = x; p.y = y; p.z = z; c.points.push_back(p); };
    for (int i = 0; i < 30000; ++i) { add(room, u(rng), u(rng), nz(rng)); add(room, u(rng), u(rng), 5.f + nz(rng)); }
    for (int i = 0; i < 8000; ++i) {
        add(room, 15.f + nz(rng), u(rng), h(rng)); add(room, -15.f + nz(rng), u(rng), h(rng));
        add(room, u(rng), 15.f + nz(rng), h(rng)); add(room, u(rng), -15.f + nz(rng), h(rng));
        add(room, 4.f + nz(rng), s(rng), h(rng)); add(room, s(rng), -6.f + nz(rng), h(rng));  // two inner walls: x / y observable
    }
    const float shifts[3][2] = {{0.2f, -0.1f}, {-0.15f, 0.25f}, {0.05f, 0.05f}};
    Cloud src[3], empty;
    for (int k = 0; k < 3; ++k)
        for (size_t i = k; i < room.points.size(); i += 23) {
            PointXYZI p = room.points[i];
            p.x += shifts[k][0];
            p.y += shifts[k][1];
            src[k].points.push_back(p);
        }
    try {
        NdtPairBatch<Cloud> batch;
        batch.setResolution(1.0f);
        batch.setTransformationEpsilon(0.01);
        batch.setNeighborhoodSearchMethod(DIRECT7);
        batch.align({&src[0], &src[1], &empty, &src[2]}, {&room, &room, &room, &room});
        for (size_t p = 0; p < batch.size(); ++p)
            std::printf("pair %zu status %d converged %d iters %d fitness %.5f tx %.4f ty %.4f\n", p, batch.status(p), (int)batch.hasConverged(p),
                        batch.getFinalNumIteration(p), batch.getFitnessScore(p), batch.getFinalTransformation(p)[12], batch.getFinalTransformation(p)[13]);
        if (batch.status(2) != B200_ERR_ARG || batch.hasConverged(2)) return 4;
        for (int k = 0; k < 3; ++k) {
            const size_t p = k < 2 ? k : 3;
            const float* T = batch.getFinalTransformation(p);
            if (!batch.hasConverged(p) || std::fabs(T[12] + shifts[k][0]) > 0.02f || std::fabs(T[13] + shifts[k][1]) > 0.02f ||
                !(batch.getFitnessScore(p) < 0.01))
                return 5;
        }
    } catch (const std::exception& e) {
        std::printf("FAILED LOUDLY: %s\n", e.what());
        return 10;
    }
    std::printf("ndt pairs adaptor ok\n");
    return 0;
}
