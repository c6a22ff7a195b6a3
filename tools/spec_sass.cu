// Offline look at the specialised state kernel for the iiwa structure (no GPU needed):
//   nvcc -std=c++17 -o /tmp/spec_sass tools/spec_sass.cu -ldl && /tmp/spec_sass /tmp/spec.cubin && cuobjdump -sass /tmp/spec.cubin
#include <cstdio>
#include "../include/stomp_b200.h"
#include "../motion_planners_b200/csrc/state_codegen.hpp"
using namespace stomp_b200;
int main(int argc, char** argv)
{
    RobotParams r;
    std::memset(&r, 0, sizeof r);
    const bool dual = getenv("DUAL") != nullptr;      // BASELINE config 5: two arms, 8 grasped-object spheres on the first tip
    r.num_joints = 7;
    const int kinds[7] = {kAxisZ, kAxisY, kAxisZ, kAxisNegY, kAxisZ, kAxisY, kAxisZ};
    const int omask[7] = {0, 5, 0, 5, 0, 4, 0};
    const int nsph[7] = {3, 3, 3, 3, 3, 2, 3};
    const int smask[20] = {4, 4, 4, 0, 6, 6, 4, 4, 4, 0, 6, 6, 4, 4, 4, 0, 4, 4, 4, 4};
    int s = 0;
    for (int d = 0; d < 7; ++d) {
        r.joint[d].axis_kind = kinds[d]; r.joint[d].o_mask = omask[d]; r.joint[d].fixed_rot_identity = 1;
        r.joint[d].parent = d - 1;
        r.sphere_begin[d] = s;
        for (int k = 0; k < nsph[d]; ++k, ++s) r.sphere[s].mask = smask[s];
    }
    if (dual) {
        for (int k = 0; k < 8; ++k, ++s) r.sphere[s].mask = 7;                      // object spheres: full offsets
        r.sphere_begin[7] = s;
        for (int d = 0; d < 7; ++d) {
            r.joint[7 + d].axis_kind = kinds[d]; r.joint[7 + d].o_mask = d == 0 ? 2 : omask[d]; r.joint[7 + d].fixed_rot_identity = 1;
            r.joint[7 + d].parent = d == 0 ? -1 : 7 + d - 1;
            r.sphere_begin[7 + d] = s;
            for (int k = 0; k < nsph[d]; ++k, ++s) r.sphere[s].mask = smask[r.sphere_begin[d] + k < 20 ? (r.sphere_begin[7 + d] - r.sphere_begin[7]) + k : 0];
        }
        r.num_joints = 14;
        r.joint[0].o_mask = 2;                                                         // bases at y = -+0.4
    }
    for (int d = r.num_joints; d <= STOMP_B200_MAX_DIMS; ++d) r.sphere_begin[d] = s;
    r.num_spheres = s;
    codegen::StateKernelOptions opt;
    opt.magic_floor = !getenv("CVT");
    opt.inside_grid = !getenv("CLAMP");
    if (getenv("LAG")) opt.compare_lag = atoi(getenv("LAG"));
    if (getenv("MINB")) opt.min_blocks = atoi(getenv("MINB"));
    if (getenv("BATCH")) opt.batch_sincos = atoi(getenv("BATCH"));
    if (getenv("NOTAIL")) opt.no_tail = atoi(getenv("NOTAIL")) != 0;
    if (getenv("LANES")) opt.rollout_lanes = true;
    if (getenv("STATIC")) opt.hoist_static = atoi(getenv("STATIC")) != 0;
    codegen::SelfPairStructure sp;
    if (dual && getenv("PAIRS")) {      // the sphere-pair rule inside the kernel: every sphere of the first arm (object included) against every one of the second
        std::vector<int> link_of((size_t)s, 0);
        for (int d = 0; d < r.num_joints; ++d) for (int k = r.sphere_begin[d]; k < r.sphere_begin[d + 1]; ++k) link_of[k] = d;
        for (int i = 0; i < r.sphere_begin[7]; ++i)
            for (int j = r.sphere_begin[7]; j < s; ++j) { sp.i.push_back(i); sp.j.push_back(j); }
        std::vector<size_t> order(sp.i.size());
        for (size_t p = 0; p < order.size(); ++p) order[p] = p;
        std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) {
            return std::make_pair(link_of[sp.i[a]], link_of[sp.j[a]]) < std::make_pair(link_of[sp.i[b]], link_of[sp.j[b]]); });
        codegen::SelfPairStructure sorted;
        for (size_t p : order) {
            const int la = link_of[sp.i[p]], lb = link_of[sp.j[p]];
            if (sorted.blocks.empty() || sorted.blocks.back().la != la || sorted.blocks.back().lb != lb)
                sorted.blocks.push_back({la, lb, (int)sorted.i.size(), (int)sorted.i.size()});
            sorted.i.push_back(sp.i[p]); sorted.j.push_back(sp.j[p]);
            sorted.blocks.back().end = (int)sorted.i.size();
        }
        sp = sorted;
        opt.self = &sp; opt.no_tail = true;
        std::printf("%zu pairs in %zu link-pair blocks\n", sp.i.size(), sp.blocks.size());
    }
    const std::string src = codegen::generate_state_kernel_source(r, opt);
    std::vector<char> cubin; std::string log, err;
    if (!codegen::compile_to_cubin(src, cubin, log, err)) { std::fprintf(stderr, "%s\n", err.c_str()); return 1; }
    if (argc > 2) { FILE* f = std::fopen(argv[2], "w"); std::fputs(src.c_str(), f); std::fclose(f); }
    FILE* f = std::fopen(argc > 1 ? argv[1] : "/tmp/spec.cubin", "wb");
    std::fwrite(cubin.data(), 1, cubin.size(), f); std::fclose(f);
    std::printf("%zu bytes; log: %s\n", cubin.size(), log.c_str());
    return 0;
}
