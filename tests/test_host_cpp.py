"""The C++ host mirror of the reference's planner API (include/, motion_planners_b200/host/):
host-side logic on the CPU, and the re-targeted test_motion_planners on the GPU."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HOST = os.path.join(ROOT, "motion_planners_b200", "host")


def _build():
    subprocess.run(["make", "-C", os.path.join(ROOT, "motion_planners_b200", "csrc"), "-s"], check=True)
    subprocess.run(["make", "-C", HOST, "-s"], check=True)


def test_host_logic_cpp(tmp_path):
    _build()
    exe = str(tmp_path / "host_logic_test")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "host_logic_test.cpp"), "-o", exe,
                    "-L" + os.path.join(ROOT, "motion_planners_b200"), "-lmotion_planners_b200", "-lstomp_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "motion_planners_b200")], check=True)
    out = subprocess.run([exe, os.path.join(ROOT, "test"), str(tmp_path)], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout + out.stderr
    for name in ("yaml_and_stomp_config", "robot_model", "meshes", "planner_api", "policy"):
        assert f"ok {name}" in out.stdout


@pytest.mark.gpu
def test_test_motion_planners_finds_a_path():
    """Config 1: the reference's demo query through MotionPlanners -> PlannerFactory -> StompPlanner::solve."""
    _build()
    exe = os.path.join(ROOT, "test", "test_motion_planners")
    out = subprocess.run([exe, os.path.join(ROOT, "test")], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    assert "Path Found" in out.stdout
    assert "Number of timestep :20. Number of joints = 7" in out.stdout
    def _floats(line):
        try:
            return [float(x) for x in line.split()]
        except ValueError:
            return []
    rows = [r for r in map(_floats, out.stdout.splitlines()) if len(r) == 7]
    assert len(rows) == 20
    first, last = rows[0], rows[-1]
    start = [0.5, 0.5, 0.5, -1.5, 0.5, 0.5, 0.5]
    goal = [-1.5, -1.5, -1.5, 1.5, -1.5, -1.5, -0.5]
    assert max(abs(a - b) for a, b in zip(first, start)) < 0.35
    assert max(abs(a - b) for a, b in zip(last, goal)) < 0.35


@pytest.mark.gpu
def test_requests_by_joint_name_and_late_scene_changes(tmp_path):
    """MotionPlanners facade: start / goal assembled by joint name, NaN / missing / out-of-limit values refused, and a
    world object added after initialize() reaches the validity checks and the next solve (tests/cpp/scene_and_request_test.cpp)."""
    _build()
    exe = str(tmp_path / "scene_and_request_test")
    subprocess.run(["/usr/bin/g++", "-std=c++17", "-O1", "-I" + os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "cpp", "scene_and_request_test.cpp"), "-o", exe,
                    "-L" + os.path.join(ROOT, "motion_planners_b200"), "-lmotion_planners_b200", "-lstomp_b200",
                    "-Wl,-rpath," + os.path.join(ROOT, "motion_planners_b200")], check=True)
    out = subprocess.run([exe, os.path.join(ROOT, "test"), str(tmp_path)], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stdout + out.stderr
    for name in ("request_by_name", "refused_requests", "scene_change_reaches_the_validity_checks",
                 "scene_change_reaches_the_next_solve", "world_objects_meshes_octomap_grasp"):
        assert f"ok {name}" in out.stdout
