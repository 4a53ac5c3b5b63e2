// Compiles the relocalization adaptor (b200host::NormalDistributionsTransform::relocalizeRefine, host/ndt_gpu.hpp) against the C
// ABI and runs it (used by tests/test_reloc_refine_cpu.py and tests/test_gpu_reloc_refine.py).  Without a GPU it must fail loudly
// at the first call; with one it relocalizes a drifted copy of a small room from a 3 x 3 grid of starts around the truth.
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
    auto room = std::make_shared<Cloud>();
    auto add = [&](Cloud& c, float x, float y, float z) { PointXYZI p{}; p.x = x; p.y = y; p.z = z; c.points.push_back(p); };
    for (int i = 0; i < 30000; ++i) { add(*room, u(rng), u(rng), nz(rng)); add(*room, u(rng), u(rng), 5.f + nz(rng)); }
    for (int i = 0; i < 8000; ++i) {
        add(*room, 15.f + nz(rng), u(rng), h(rng)); add(*room, -15.f + nz(rng), u(rng), h(rng));
        add(*room, u(rng), 15.f + nz(rng), h(rng)); add(*room, u(rng), -15.f + nz(rng), h(rng));
        add(*room, 4.f + nz(rng), s(rng), h(rng)); add(*room, s(rng), -6.f + nz(rng), h(rng));  // two inner walls: x / y observable
    }
    const float shift[2] = {0.3f, -0.2f};  // the scan is the room seen from (-0.3, 0.2): its pose is a translation by +shift
    auto scan = std::make_shared<Cloud>();
    for (size_t i = 0; i < room->points.size(); i += 23) {
        PointXYZI p = room->points[i];
        p.x -= shift[0];
        p.y -= shift[1];
        scan->points.push_back(p);
    }
    std::vector<float> grid;  // 3 x 3 starts, 0.5 m apart, around the origin
    for (int iy = -1; iy <= 1; ++iy)
        for (int ix = -1; ix <= 1; ++ix) {
            float T[16] = {1, 0, 0, 0, 0, 1, 0, 0, 0, 0, 1, 0, 0.5f * ix, 0.5f * iy, 0, 1};
            grid.insert(grid.end(), T, T + 16);
        }
    try {
        NormalDistributionsTransform<Cloud> ndt;
        ndt.setResolution(1.0f);
        ndt.setTransformationEpsilon(0.01);
        ndt.setInputTarget(room);
        ndt.setInputSource(scan);
        std::vector<b200_reloc_candidate> cands;
        bool converged = false;
        const int64_t best = ndt.relocalizeRefine(nullptr, grid.data(), 9, 0, 1, 4, cands, &converged);
        std::printf("best %lld converged %d candidates %zu\n", (long long)best, (int)converged, cands.size());
        const b200_reloc_candidate* w = nullptr;
        for (const auto& c : cands) {
            std::printf("hyp %lld score %.4f status %d tx %.4f ty %.4f\n", (long long)c.hypothesis, c.initial_score, c.refined.status,
                        c.refined.final16[12], c.refined.final16[13]);
            if (c.hypothesis == best) w = &c;
        }
        if (cands.size() != 4 || !converged || !w) return 4;
        if (std::fabs(w->refined.final16[12] - shift[0]) > 0.02f || std::fabs(w->refined.final16[13] - shift[1]) > 0.02f) return 5;
    } catch (const std::exception& e) {
        std::printf("FAILED LOUDLY: %s\n", e.what());
        return 10;
    }
    std::printf("relocalization adaptor ok\n");
    return 0;
}
