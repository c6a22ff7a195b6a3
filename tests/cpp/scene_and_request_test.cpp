// GPU test of the facade around the hot path (reference src/MotionPlanners.cpp:91-219,416-460): planning requests are
// assembled by joint NAME, NaN / missing / out-of-limit values are refused, and a world object added after
// initialize() takes effect at once — in the validity checks and in the next solve (the engines rebuild their distance
// field on the device when the scene revision changes).
//   ./scene_and_request_test <absolute path to the test folder>
#include <cmath>
#include <cstdio>
#include <iostream>

#include <motion_planners/MotionPlanners.hpp>
#include <robot_model/MeshTools.hpp>

using namespace motion_planners;

#define CHECK(cond) do { if (!(cond)) { std::printf("FAILED %s:%d: %s\n", __FILE__, __LINE__, #cond); return 1; } } while (0)

static base::samples::Joints joints(const std::vector<std::string>& names, const std::vector<double>& values)
{
    base::samples::Joints j;
    j.names = names;
    j.elements.resize(values.size());
    for (size_t i = 0; i < values.size(); ++i) j.elements[i].position = values[i];
    return j;
}

int main(int argc, char** argv)
{
    if (argc != 3) return 2;
    const std::string dir = argv[1], scratch = argv[2];   // scratch: a directory of this run's own for the files it writes
    Config config;
    config.planner_config.robot_model_config.urdf_file = dir + "/data/iiwa_chain.urdf";
    config.planner_config.robot_model_config.planning_group_name = "manipulator";
    config.planner_config.robot_model_config.base_link = "base_link";
    config.planner_config.robot_model_config.tip_link = "link_7";
    config.planner_config.robot_model_config.spheres_file = dir + "/data/iiwa_spheres.yml";
    config.planner_config.robot_model_config.environment_file = dir + "/data/environment.yml";
    config.planner_config.planner_specific_config = dir + "/config/stomp.yml";
    config.planner_config.planner = STOMP;
    MotionPlanners planner(config);
    PlannerStatus status;
    CHECK(planner.initialize(status));

    const std::vector<std::string> names = {"joint_a1", "joint_a2", "joint_a3", "joint_a4", "joint_a5", "joint_a6", "joint_a7"};
    const std::vector<double> start = {0.5, 0.5, 0.5, -1.5, 0.5, 0.5, 0.5}, goal = {-1.5, -1.5, -1.5, 1.5, -1.5, -1.5, -0.5};

    // ---- by name: reversed order plus a joint that is not in the planning group ----
    std::vector<std::string> rnames(names.rbegin(), names.rend());
    std::vector<double> rstart(start.rbegin(), start.rend()), rgoal(goal.rbegin(), goal.rend());
    rnames.push_back("gripper_finger"); rstart.push_back(0.01); rgoal.push_back(0.02);
    CHECK(planner.assignPlanningRequest(joints(rnames, rstart), joints(rnames, rgoal), status));
    CHECK(status.statuscode == PlannerStatus::PLANNING_REQUEST_SUCCESS);
    planner.setStartAndGoal();
    base::JointsTrajectory initial = planner.planner_->getInitialTrajectory();
    for (int d = 0; d < 7; ++d) {
        CHECK(initial.names[d] == names[d]);
        CHECK(initial.elements[d].front().position == start[d]);
        CHECK(std::fabs(initial.elements[d].back().position - goal[d]) < 1e-12);
    }
    std::puts("ok request_by_name");

    // ---- refused requests ----
    {
        std::vector<double> bad = start;
        bad[2] = NAN;
        CHECK(!planner.assignPlanningRequest(joints(names, bad), joints(names, goal), status));
        CHECK(status.statuscode == PlannerStatus::START_JOINTANGLES_NOT_AVAILABLE);
        bad = goal; bad[5] = NAN;
        CHECK(!planner.assignPlanningRequest(joints(names, start), joints(names, bad), status));
        CHECK(status.statuscode == PlannerStatus::GOAL_JOINTANGLES_NOT_AVAILABLE);
        std::vector<std::string> six(names.begin(), names.end() - 1);
        CHECK(!planner.assignPlanningRequest(joints(six, std::vector<double>(start.begin(), start.end() - 1)), joints(names, goal), status));
        CHECK(status.statuscode == PlannerStatus::START_JOINTANGLES_NOT_AVAILABLE);
        bad = start; bad[1] = 2.5;      // limit of joint_a2 is 2.0942
        CHECK(!planner.assignPlanningRequest(joints(names, bad), joints(names, goal), status));
        CHECK(status.statuscode == PlannerStatus::INVALID_START_STATE);
        bad = goal; bad[6] = -3.2;
        CHECK(!planner.assignPlanningRequest(joints(names, start), joints(names, bad), status));
        CHECK(status.statuscode == PlannerStatus::INVALID_GOAL_STATE);
        CHECK(!planner.assignPlanningRequest(base::samples::Joints(), joints(names, goal), status));
        CHECK(status.statuscode == PlannerStatus::START_JOINTANGLES_NOT_AVAILABLE);
    }
    std::puts("ok refused_requests");

    // ---- solve, then change the world ----
    CHECK(planner.assignPlanningRequest(joints(names, start), joints(names, goal), status));
    planner.setStartAndGoal();
    base::JointsTrajectory solution;
    double seconds = 0.0;
    CHECK(planner.solve(solution, status, seconds) && status.statuscode == PlannerStatus::PATH_FOUND);
    std::shared_ptr<robot_model::RobotModel> robot = planner.getRobotModel();
    const unsigned long rev0 = robot->sceneRevision();
    // a ball around the tool at the goal configuration: the goal, free a moment ago, is now in collision
    robot_model::Obstacle ball;
    ball.kind = 0; ball.name = "late_ball";
    {
        // tool position at the goal from the solution's last state: put the ball on a state the robot provably occupies
        double cost = 0.0;
        robot->updateJointGroup(joints(names, goal));
        CHECK(robot->isStateValid(cost));
    }
    // the blocker of environment.yml sits at (-0.17, 0.03, 1.31) r 0.15 on the straight line; a large ball at the same
    // place reaches the arm at the goal configuration as well
    ball.centre[0] = -0.17; ball.centre[1] = 0.03; ball.centre[2] = 1.31; ball.size[0] = ball.size[1] = ball.size[2] = 1.2;
    robot->addObstacle(ball);
    CHECK(robot->sceneRevision() == rev0 + 1);
    CHECK(!planner.assignPlanningRequest(joints(names, start), joints(names, goal), status));
    CHECK(status.statuscode == PlannerStatus::START_STATE_IN_COLLISION || status.statuscode == PlannerStatus::GOAL_STATE_IN_COLLISION);
    CHECK(robot->removeObstacle("late_ball") && !robot->removeObstacle("late_ball"));
    CHECK(planner.assignPlanningRequest(joints(names, start), joints(names, goal), status));
    std::puts("ok scene_change_reaches_the_validity_checks");

    // a wall across the solved path: every state of the OLD solution that it cuts must be gone from the new one
    robot_model::Obstacle wall;
    wall.kind = 1; wall.name = "late_wall";
    wall.centre[0] = 0.0; wall.centre[1] = 0.75; wall.centre[2] = 0.9; wall.size[0] = 0.6; wall.size[1] = 0.08; wall.size[2] = 0.25;
    robot->addObstacle(wall);
    auto colliding_states = [&](const base::JointsTrajectory& traj) {
        int n = 0;
        for (size_t t = 0; t < traj.getTimeSteps(); ++t) {
            std::vector<double> q(7);
            for (int d = 0; d < 7; ++d) q[d] = traj.elements[d][t].position;
            double cost = 0.0;
            robot->updateJointGroup(joints(names, q));
            if (!robot->isStateValid(cost)) ++n;
        }
        return n;
    };
    const int old_hits = colliding_states(solution);
    if (planner.assignPlanningRequest(joints(names, start), joints(names, goal), status)) {
        planner.setStartAndGoal();
        base::JointsTrajectory second;
        const bool found = planner.solve(second, status, seconds);
        const int new_hits = colliding_states(second);
        std::printf("old solution: %d states inside the late wall; new solve: found=%d, %d states in collision\n", old_hits, (int)found, new_hits);
        // the planner's own verdict and the validity engine agree about the new world
        CHECK(found == (new_hits == 0) || !found);
        if (found) CHECK(new_hits == 0);
    }
    std::puts("ok scene_change_reaches_the_next_solve");
    CHECK(robot->removeObstacle("late_wall"));

    // world objects as the reference's callers hand them in (MotionPlanners::handleCollisionObjectInWorld, updateOctomap): a mesh
    // (STL), a cylinder and octomap leaves go through the device voxeliser + distance transform (stomp_b200_build_sdf_scene)
    {
        auto state_valid = [&](const std::vector<double>& q) {
            double cost = 0.0;
            robot->updateJointGroup(joints(names, q));
            return robot->isStateValid(cost);
        };
        CHECK(state_valid(start));
        // where is the arm at `start`?  put objects on the tip: the last sphere's centre from a probe engine is not exposed,
        // so use a leaf / mesh large enough around the known reach of the start pose: the blocker's place is on the straight
        // line, the arm at `start` passes near (0.25, 0.2, 0.9)
        std::vector<double> crate;
        const double zero[3] = {0, 0, 0}, half[3] = {0.9, 0.9, 0.9};
        robot_model::appendBoxMesh(zero, half, crate);         // a crate that swallows most of the workspace above the base
        const std::string stl = scratch + "/crate.stl";
        {
            FILE* f = std::fopen(stl.c_str(), "wb");
            char header[80] = "crate"; std::fwrite(header, 1, 80, f);
            const unsigned n = (unsigned)(crate.size() / 9); std::fwrite(&n, 4, 1, f);
            for (unsigned i = 0; i < n; ++i) {
                float rec[12] = {0, 0, 0};
                for (int k = 0; k < 9; ++k) rec[3 + k] = (float)crate[i * 9 + k];
                std::fwrite(rec, 4, 12, f);
                const unsigned short attr = 0; std::fwrite(&attr, 2, 1, f);
            }
            std::fclose(f);
        }
        ModelObject mesh;
        mesh.operation = collision_detection::ADD; mesh.model_type = collision_detection::MESH;
        mesh.object_name = "crate"; mesh.object_path = stl;
        mesh.relative_pose.position = base::Vector3d(0.0, 0.0, 1.2);
        CHECK(planner.handleCollisionObjectInWorld(mesh));
        CHECK(!state_valid(start));                                   // the solid crate (interior filled) holds the arm
        mesh.operation = collision_detection::REMOVE;
        CHECK(planner.handleCollisionObjectInWorld(mesh) && state_valid(start));
        ModelObject cyl;
        cyl.operation = collision_detection::ADD; cyl.model_type = collision_detection::PRIMITIVES; cyl.object_name = "column";
        cyl.primitive_object.primitive_type = collision_detection::CYLINDER; cyl.primitive_object.radius = 1.0; cyl.primitive_object.height = 1.6;
        cyl.relative_pose.position = base::Vector3d(0.0, 0.0, 1.0);
        CHECK(planner.handleCollisionObjectInWorld(cyl) && !state_valid(start));
        cyl.operation = collision_detection::REMOVE;
        CHECK(planner.handleCollisionObjectInWorld(cyl) && state_valid(start));
        OccupiedLeaves leaves;
        for (int i = -4; i <= 4; ++i) for (int j = -4; j <= 4; ++j) for (int k = 1; k <= 9; ++k) {
            leaves.centres.push_back(0.2 * i); leaves.centres.push_back(0.2 * j); leaves.centres.push_back(0.2 * k); leaves.sizes.push_back(0.2);
        }
        planner.updateOctomap(leaves);
        CHECK(!state_valid(start));
        planner.updateOctomap(OccupiedLeaves());
        CHECK(state_valid(start));
        // a grasp object: its spheres ride on the tip link; a long rod held at the tip reaches the floor obstacle the bare arm clears
        ModelObject rod;
        rod.operation = collision_detection::ADD; rod.model_type = collision_detection::PRIMITIVES; rod.object_name = "rod";
        rod.primitive_object.primitive_type = collision_detection::BOX; rod.primitive_object.dimensions = base::Vector3d(0.05, 0.05, 3.0);
        const size_t spheres_before = robot->spheres().size();
        CHECK(planner.handleGraspObject(rod) && robot->spheres().size() > spheres_before);
        robot_model::Obstacle shell;       // a thick spherical band far out: only the 1.5 m rod ends can be in it
        shell.kind = 1; shell.name = "far_wall"; shell.centre[0] = 0.0; shell.centre[1] = 0.0; shell.centre[2] = -1.2; shell.size[0] = 1.5; shell.size[1] = 1.5; shell.size[2] = 0.25;
        robot->addObstacle(shell);
        const bool with_rod = state_valid(start);
        rod.operation = collision_detection::REMOVE;
        CHECK(planner.handleGraspObject(rod) && robot->spheres().size() == spheres_before);
        const bool without_rod = state_valid(start);
        std::printf("far wall: valid with the rod %d, without %d\n", (int)with_rod, (int)without_rod);
        CHECK(without_rod);
        robot->removeObstacle("far_wall");
    }
    std::puts("ok world_objects_meshes_octomap_grasp");
    return 0;
}
