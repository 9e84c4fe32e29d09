// Host build of the union-find of csrc/sfm_track_build.cuh (tb_find, tb_hook) for tests/test_track_build_oracle.py:
// the hook runs on several CPU threads at once over interleaved edges, then the compress pass, as the kernels do.
#include <thread>
#include <vector>

#include "../structure_from_motion_b200/csrc/sfm_track_build.cuh"

// edges int32[E][2] of global ids in [0, N); label int32[N] receives each feature's root (its component's minimum).
extern "C" void tb_components(int N, long long E, const int* edges, int threads, int* label) {
    std::vector<int> parent(N);
    for (int g = 0; g < N; ++g) parent[g] = g;
    std::vector<std::thread> pool;
    for (int w = 0; w < threads; ++w)
        pool.emplace_back([&, w] {
            for (long long e = w; e < E; e += threads) sfm::tb_hook(parent.data(), edges[2 * e], edges[2 * e + 1]);
        });
    for (auto& t : pool) t.join();
    pool.clear();
    for (int w = 0; w < threads; ++w)
        pool.emplace_back([&, w] {
            for (int g = w; g < N; g += threads) label[g] = sfm::tb_find(parent.data(), g);
        });
    for (auto& t : pool) t.join();
}

extern "C" int tb_view_of(const long long* off, int V, long long g) { return sfm::tb_view_of(off, V, g); }
