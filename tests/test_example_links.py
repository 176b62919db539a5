"""SURVEY 8(b) / north star "MonoSlamSceneLib1 links unchanged": the reference's own examples/MonoSlamSceneLib1.cpp,
compiled WHERE IT LIES and unmodified, against the host shim (scenelib2_b200/host) and libsl2b200.so.  Pangolin, GLUT
and the two GUI mouse handlers are header / symbol stand-ins under tests/example_standins (test infrastructure only).
Every member the example touches -- camera_->{width_, height_, fku_, fkv_, centre_}, graphic_tool_->Draw3dScene /
DrawAR, frame_grabber_->GetFrame, GoOneStep, InitialiseFeature, InitialiseAutoFeature, print_robot_state,
delete_feature, SavePatch, SceneLib2::Frame -- therefore has to exist on the shim with a compatible signature."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_unchanged_example_compiles_and_links_against_the_shim(tmp_path):
    import __graft_entry__ as g
    from oracle import pyoracle
    g.build()
    # the example is not part of this repository: it is compiled from the SceneLib2 tree build() built oracle/_ref from
    src = pyoracle.scenelib2_src()
    if src is None:
        pytest.skip("oracle/_ref not built from a SceneLib2 source tree")
    example = os.path.join(src, "examples", "MonoSlamSceneLib1.cpp")
    host = os.path.join(ROOT, "scenelib2_b200", "host")
    lib = os.path.join(ROOT, "scenelib2_b200")
    st = os.path.join(ROOT, "tests", "example_standins")
    exe = str(tmp_path / "MonoSlamSceneLib1")
    cmd = ["g++", "-std=c++17", "-O0", "-pthread", "-I", st, "-I", host, "-I", os.path.join(src, "scenelib2"),
           example, os.path.join(st, "gui_stubs.cpp"), "-o", exe,
           "-L", host, "-lscenelib2_b200_host", "-L", lib, "-lsl2b200",
           "-Wl,-rpath," + host, "-Wl,-rpath," + lib]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    # every symbol the example needs resolved against the shim library (nothing supplied by the stand-ins but the GUI)
    nm = subprocess.run(["nm", "-C", "--undefined-only", exe], capture_output=True, text=True).stdout
    for sym in ("SceneLib2::MonoSLAM::Init", "SceneLib2::MonoSLAM::GoOneStep", "SceneLib2::MonoSLAM::InitialiseFeature",
                "SceneLib2::MonoSLAM::InitialiseAutoFeature", "SceneLib2::MonoSLAM::SavePatch",
                "SceneLib2::MonoSLAM::delete_feature", "SceneLib2::MonoSLAM::print_robot_state",
                "SceneLib2::GraphicTool::Draw3dScene", "SceneLib2::GraphicTool::DrawAR",
                "SceneLib2::FrameGrabber::GetFrame"):
        assert sym in nm, sym
    # it starts: without a GPU the shim refuses loudly in Init (no CPU fallback), with one it needs the cfg of the
    # reference's data directory -- either way the dynamic linker found both libraries
    run = subprocess.run([exe], capture_output=True, text=True, cwd=str(tmp_path))
    assert "error while loading shared libraries" not in run.stderr
