// Host-side logic of the C++ drop-in (no GPU needed): YAML subset, StompConfig parsing, URDF chain,
// spheres, SDF builder, CovariantMovementPrimitive, PlannerFactory / StompPlanner API up to solve().
// Prints one "ok <name>" line per check; exits non-zero on the first failure.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <iostream>
#include <string>

#include <PlannerFactory.hpp>
#include <motion_planners/MotionPlanners.hpp>
#include <robot_model/MeshTools.hpp>
#include <vector>
#include <stomp_b200.h>

#define CHECK(cond)                                                                  \
    do {                                                                             \
        if (!(cond)) {                                                               \
            std::fprintf(stderr, "FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond);   \
            std::exit(1);                                                            \
        }                                                                            \
    } while (0)

using namespace motion_planners;

int main(int argc, char** argv)
{
    CHECK(argc == 3);
    const std::string test_dir = argv[1], scratch = argv[2];   // scratch: a directory of this run's own for the files it writes

    // ---- YAML subset + StompConfig (reference HandleStompConfig.cpp:7-63, test/config/stomp.yml) ----
    YAML::Node cfg;
    loadConfigFile(test_dir + "/config/stomp.yml", cfg);
    CHECK(cfg["stomp"] && cfg["debug"] && !cfg["nope"]);
    stomp::StompConfig sc = handle_stomp_config::getStompConfig(cfg["stomp"]);
    CHECK(sc.max_rollouts_ == 50 && sc.min_rollouts_ == 5 && sc.num_rollouts_per_iteration_ == 10);
    CHECK(sc.num_iterations_ == 30 && sc.num_time_steps_ == 20 && sc.num_dimensions_ == 7);
    CHECK(sc.movement_duration_ == 5.0 && sc.control_cost_weight_ == 0.001 && sc.min_cost_improvement_ == 0.01);
    CHECK(sc.noise_stddev_.size() == 7 && sc.noise_stddev_[2] == 0.5 && sc.noise_decay_[6] == 1.0 && sc.noise_min_stddev_[0] == 0.01);
    CHECK(sc.use_noise_adaptation_ && !sc.use_openmp_ && sc.seed_ == 2024);
    stomp::DebugConfig dc = handle_stomp_config::getDebugConfig(cfg["debug"]);
    CHECK(dc.output_dir_ == "./debug_data" && !dc.save_noisy_trajectories_);
    // ints written as doubles fall back through getValue<int,double> (AbstractPlanner.hpp:32-50)
    YAML::Node n = YAML::Load("a: 5.0\nb: [1, 2.5, 3]\nc:\n  d: true\n  e: 'text'\nf:\n  - 1\n  - 2\n");
    CHECK((getValue<int, double>(n, "a") == 5) && n["b"].size() == 3 && n["b"][1].as<double>() == 2.5);
    CHECK(n["c"]["d"].as<bool>() && n["c"]["e"].as<std::string>() == "text" && n["f"].size() == 2);
    bool threw = false;
    try { n["c"]["e"].as<double>(); } catch (const YAML::Exception&) { threw = true; }
    CHECK(threw);
    std::puts("ok yaml_and_stomp_config");

    // ---- robot model: URDF chain, limits, spheres, obstacles, SDF ----
    robot_model::RobotModelConfig rc;
    rc.urdf_file = test_dir + "/data/iiwa_chain.urdf";
    rc.planning_group_name = "manipulator";
    rc.base_link = "base_link";
    rc.tip_link = "link_7";
    rc.spheres_file = test_dir + "/data/iiwa_spheres.yml";
    rc.environment_file = test_dir + "/data/environment.yml";
    std::shared_ptr<robot_model::RobotModel> robot(new robot_model::RobotModel(rc));
    CHECK(robot->initialization());
    CHECK(robot->chain().size() == 7 && robot->chain()[3].axis[1] == -1.0 && robot->chain()[1].origin_xyz[2] == 0.36);
    std::vector<double> lo, up;
    CHECK(robot->getJointLimits(lo, up) && lo[6] == -3.0541 && up[1] == 2.0942);
    CHECK(robot->spheres().size() == 20 && robot->spheres()[19].link == 6 && robot->spheres()[4].xyz[1] == 0.05);
    CHECK(robot->getBaseFrameName() == "base_link" && robot->getTipFrameName() == "link_7");
    CHECK(robot->obstacles().size() == 3);   // box_1 from the URDF + blocker + shelf
    const robot_model::SignedDistanceField& sdf = robot->sdf();
    CHECK(sdf.dims[0] == 64 && sdf.grid.size() == 64u * 64 * 64 && std::fabs(sdf.voxel - 3.0 / 64) < 1e-15);
    auto at = [&](double x, double y, double z) {
        int ix = (int)std::floor((x - sdf.origin[0]) / sdf.voxel), iy = (int)std::floor((y - sdf.origin[1]) / sdf.voxel),
            iz = (int)std::floor((z - sdf.origin[2]) / sdf.voxel);
        return sdf.grid[((size_t)iz * 64 + iy) * 64 + ix];
    };
    CHECK(at(0.5, 0.0, 0.5) < -0.05);          // inside box_1
    CHECK(at(-0.17, 0.03, 1.31) < -0.1);       // inside the blocker sphere
    CHECK(at(0.0, 0.0, 0.0) > 0.3);            // free space at the base
    // self collision: off by default; on -> every pair of spheres on different, not directly joined links; the SRDF's
    // disable_collisions entries remove link pairs (either order of the names)
    CHECK(robot->selfCollisionPairs().empty());
    {
        auto count_links = [&](const std::vector<std::pair<int, int> >& pairs, int a, int b) {
            int n = 0;
            for (const auto& p : pairs) n += robot->spheres()[p.first].link == a && robot->spheres()[p.second].link == b;
            return n;
        };
        robot->setSelfCollision(true);
        const auto all = robot->selfCollisionPairs();
        // spheres per link: 3 3 3 3 3 2 3 -> pairs over different links 20*19/2 - (6*3 + 1) = 171; joined links: 9*4 + 6 + 6 = 48
        CHECK(all.size() == 171u - 48u);
        CHECK(count_links(all, 0, 1) == 0 && count_links(all, 0, 2) == 9 && count_links(all, 4, 6) == 9 && count_links(all, 3, 5) == 6);
        for (const auto& p : all) CHECK(p.first < p.second);
        robot_model::RobotModelConfig rs = rc;
        rs.srdf_file = test_dir + "/data/iiwa_chain.srdf";
        rs.self_collision = true;
        robot_model::RobotModel with_srdf(rs);
        CHECK(with_srdf.initialization());
        const auto fewer = with_srdf.selfCollisionPairs();
        // removed: (0,2) (1,3) (2,4): 9 each, (3,5): 6, (4,6) written as link_7/link_5: 9
        CHECK(fewer.size() == all.size() - 42u);
        CHECK(count_links(fewer, 0, 2) == 0 && count_links(fewer, 4, 6) == 0 && count_links(fewer, 0, 3) == 9 && count_links(fewer, 1, 6) == 9);
        robot->setSelfCollision(false);
    }
    std::puts("ok robot_model");

    // ---- meshes: STL input, sphere fitting, grasp objects, world objects (SURVEY 8f rank 2) ----
    {
        // a 0.1 x 0.14 x 0.6 box as a binary and as an ASCII STL
        std::vector<double> box;
        const double bc[3] = {0.02, -0.01, 0.3}, bh[3] = {0.05, 0.07, 0.3};
        robot_model::appendBoxMesh(bc, bh, box);
        CHECK(box.size() == 12u * 9u);
        const std::string bin = scratch + "/box.stl", asc = scratch + "/box_ascii.stl";
        {
            FILE* f = std::fopen(bin.c_str(), "wb");
            char header[80] = "solid binary box";     // a binary file that starts with "solid": recognised by its size
            std::fwrite(header, 1, 80, f);
            const unsigned n = 12; std::fwrite(&n, 4, 1, f);
            for (unsigned i = 0; i < n; ++i) {
                float rec[12] = {0, 0, 0};
                for (int k = 0; k < 9; ++k) rec[3 + k] = (float)box[i * 9 + k];
                std::fwrite(rec, 4, 12, f);
                const unsigned short attr = 0; std::fwrite(&attr, 2, 1, f);
            }
            std::fclose(f);
            f = std::fopen(asc.c_str(), "w");
            std::fprintf(f, "solid box\n");
            for (unsigned i = 0; i < n; ++i) {
                std::fprintf(f, " facet normal 0 0 0\n  outer loop\n");
                for (int k = 0; k < 3; ++k) std::fprintf(f, "   vertex %.9g %.9g %.9g\n", box[i * 9 + 3 * k], box[i * 9 + 3 * k + 1], box[i * 9 + 3 * k + 2]);
                std::fprintf(f, "  endloop\n endfacet\n");
            }
            std::fprintf(f, "endsolid box\n");
            std::fclose(f);
        }
        std::vector<double> from_bin, from_asc;
        const double shift[3] = {1.0, 0.0, -1.0}, scale[3] = {2.0, 1.0, 1.0};
        CHECK(robot_model::loadStl(bin, from_bin) && from_bin.size() == box.size());
        CHECK(robot_model::loadStl(asc, from_asc, scale, shift) && from_asc.size() == box.size());
        for (size_t i = 0; i < box.size(); ++i) {
            CHECK(std::fabs(from_bin[i] - box[i]) < 1e-6);
            CHECK(std::fabs(from_asc[i] - (box[i] * scale[i % 3] + shift[i % 3])) < 1e-6);
        }
        std::vector<double> none;
        CHECK(!robot_model::loadStl(scratch + "/no_such_file.stl", none) && none.empty());
        // sphere fit: slabs along the long (z) axis, every vertex covered, radii close to the slab's half diagonal
        const auto fit = robot_model::fitSpheres(box, 8, 0.0);
        CHECK(fit.size() >= 3 && fit.size() <= 8);
        for (size_t v = 0; v < box.size() / 3; ++v) {
            bool covered = false;
            for (const auto& sp : fit) {
                double d2 = 0; for (int a = 0; a < 3; ++a) d2 += (box[3 * v + a] - sp.xyz[a]) * (box[3 * v + a] - sp.xyz[a]);
                covered = covered || std::sqrt(d2) <= sp.radius;
            }
            CHECK(covered);
        }
        for (const auto& sp : fit) { CHECK(sp.radius < 0.2 && std::fabs(sp.xyz[0] - 0.02) < 1e-9 && std::fabs(sp.xyz[1] + 0.01) < 1e-9); }
        CHECK(robot_model::fitSpheres(box, 1, 0.01).size() == 1);
        // grasp object: its spheres join the tip link's, the robot revision moves, removal restores the list
        const size_t s0 = robot->spheres().size();
        const unsigned long r0 = robot->robotRevision();
        robot_model::GraspObject go;
        go.name = "bottle";
        for (const auto& sp : fit) { robot_model::CollisionSphere cs; cs.link = 0; for (int a = 0; a < 3; ++a) cs.xyz[a] = sp.xyz[a]; cs.radius = sp.radius; go.spheres.push_back(cs); }
        CHECK(robot->addGraspObject(go, "") && robot->spheres().size() == s0 + fit.size() && robot->robotRevision() > r0);
        CHECK(robot->spheres().back().link == 6);
        CHECK(!robot->addGraspObject(go, "no_such_link"));
        CHECK(robot->addGraspObject(go, "link_3") && robot->spheres().size() == s0 + fit.size());      // re-attached, not duplicated
        CHECK(robot->removeGraspObject("bottle") && robot->spheres().size() == s0 && !robot->removeGraspObject("bottle"));
        // world objects: mesh from STL, cylinder primitive, octomap leaves -> scene revision moves
        const unsigned long sr = robot->sceneRevision();
        const double pos[3] = {0.4, 0.4, 0.0};
        CHECK(robot->addMeshObstacleFromStl("crate", bin, pos) && robot->meshObstacles().size() == 1 && robot->sceneRevision() > sr);
        CHECK(robot->removeObstacle("crate") && robot->meshObstacles().empty());
        robot->setOctomapLeaves({0.3, 0.3, 0.3}, {0.1});
        robot->setOctomapLeaves({}, {});
    }
    std::puts("ok meshes");

    // ---- CovariantMovementPrimitive against the C-ABI host policy ----
    const int T = 20, D = 7, N = T + 12;
    std::vector<double> start = {0.5, 0.5, 0.5, -1.5, 0.5, 0.5, 0.5}, goal = {-1.5, -1.5, -1.5, 1.5, -1.5, -1.5, -0.5};
    std::vector<double> init((size_t)D * N), R(T * T), Rinv(T * T), L(T * T), pall((size_t)D * N), mincc((size_t)D * T);
    CHECK(stomp_b200_host_initial_trajectory(T, D, start.data(), goal.data(), init.data()) == 0);
    const double w[4] = {0, 0, 1, 0};
    CHECK(stomp_b200_host_policy(T, D, 5.0, w, init.data(), 1, R.data(), Rinv.data(), L.data(), pall.data(), mincc.data()) == 0);

    // ---- planner API up to solve() ----
    PlannerFactory factory;
    CHECK(factory.getPlannerTask(OMPL) == NULL && factory.getPlannerTask(TRAJOPT) == NULL);
    AbstractPlannerPtr planner = factory.getPlannerTask(STOMP);
    CHECK(planner && std::dynamic_pointer_cast<StompPlanner>(planner));
    CHECK(planner->initializePlanner(robot, test_dir + "/config/stomp.yml"));
    base::samples::Joints s, g;
    s.resize(7); g.resize(7);
    for (int i = 0; i < 7; ++i) {
        s.names[i] = g.names[i] = "joint_a" + std::to_string(i + 1);
        s.elements[i].position = start[i];
        g.elements[i].position = goal[i];
    }
    planner->setStartGoalTrajectory(s, g);
    base::JointsTrajectory initial = planner->getInitialTrajectory();
    CHECK(initial.getNumberOfJoints() == 7 && initial.getTimeSteps() == 20);
    for (int d = 0; d < D; ++d) {
        // getInitialTrajectory returns the linear interpolation (input_initial_trajectory_, StompPlanner.cpp:210-229)
        CHECK(initial.elements[d][0].position == start[d]);
        CHECK(std::fabs(initial.elements[d][19].position - goal[d]) < 1e-12);
        CHECK(initial.names[d] == s.names[d]);
    }
    StompPlanner* sp = static_cast<StompPlanner*>(planner.get());
    CHECK(std::fabs(sp->getMovementDeltaTime() - 5.0 / 21) < 1e-15);
    CHECK(planner->getNumOfIterationsUsed() == 0);
    std::puts("ok planner_api");

    // ---- the policy held by the planner equals the C-ABI host policy ----
    {
        stomp::CovariantMovementPrimitive cmp;
        std::vector<base::MatrixXd> dcosts(D, base::MatrixXd::Zero(N, 4));
        std::vector<base::VectorXd> traj(D, base::VectorXd::Zero(N));
        for (int d = 0; d < D; ++d)
            for (int i = 0; i < N; ++i) { dcosts[d](i, 2) = 1.0; traj[d](i) = init[(size_t)d * N + i]; }
        CHECK(cmp.initialize(T, D, 5.0, dcosts, traj) && cmp.setToMinControlCost());
        for (int d = 0; d < D; ++d)
            for (int i = 0; i < N; ++i) CHECK(cmp.parameters_all_[d](i) == pall[(size_t)d * N + i]);
        for (int i = 0; i < T * T; ++i) CHECK(cmp.R()[i] == R[i] && cmp.L()[i] == L[i]);
        base::MatrixXd acc = cmp.getDifferentiationMatrix(stomp::STOMP_ACCELERATION);
        double row = 0.0;
        for (int j = 0; j < N; ++j) row += acc(10, j);
        CHECK(std::fabs(row) < 1e-9 && acc(10, 10) < 0.0);
        dcosts[3](5, 2) = 2.0;    // per-joint weights are outside this build: rejected, not silently ignored
        CHECK(!cmp.initialize(T, D, 5.0, dcosts, traj));
    }
    std::puts("ok policy");

    // ---- without a CUDA device solve() reports a failed initialisation (no CPU fallback) ----
    int ndev_status = 0;
    {
        stomp_b200_config c;
        stomp_b200_default_config(&c);
        c.num_time_steps = 20; c.num_dimensions = 7; c.min_rollouts = c.max_rollouts = c.num_rollouts_per_iteration = 4;
        stomp_b200_engine* e = nullptr;
        ndev_status = stomp_b200_create(&c, &e);
        if (e) stomp_b200_destroy(e);
    }
    if (ndev_status == STOMP_B200_ERR_NO_DEVICE) {
        base::JointsTrajectory solution;
        PlannerStatus status;
        CHECK(!planner->solve(solution, status));
        CHECK(status.statuscode == PlannerStatus::PLANNER_INITIALISATION_FAILED);
        std::puts("ok no_device_no_fallback");
    } else {
        std::puts("ok device_present_skipping_no_device_check");
    }
    return 0;
}
