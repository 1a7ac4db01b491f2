"""The C++ drop-in adaptor (include/wso_tessendorf_adaptor.hpp) and the headless caller (examples/frame_loop.cpp):
compile checks on CPU, end-to-end run against the Python path on the GPU."""
import json
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT

EX = os.path.join(ROOT, "examples")
GXX = "/usr/bin/g++" if os.path.exists("/usr/bin/g++") else "g++"


def _build_frame_loop():
    from watersurfacerendering_b200 import build as B
    B.build()
    subprocess.check_call(["make", "-C", EX, "frame_loop"], stdout=subprocess.DEVNULL)
    return os.path.join(EX, "frame_loop")


def test_adaptor_and_caller_compile():
    exe = _build_frame_loop()
    assert os.path.exists(exe)


def test_adaptor_exposes_the_reference_interface(tmp_path):
    """Every public member the reference's caller uses (WaterSurfaceMesh.cpp:127-179, 705-741, 804-902)."""
    src = tmp_path / "iface.cpp"
    src.write_text(r'''
#include <cstring>
#include <vector>
#include "wso_tessendorf_adaptor.hpp"
static_assert(sizeof(WSTessendorf::Displacement) == 16 && sizeof(WSTessendorf::Normal) == 16, "RGBA32F texels");
float use(WSTessendorf& m, std::vector<unsigned char>& staging) {
    m.SetTileSize(WSTessendorf::s_kDefaultTileSize);
    m.SetTileLength(WSTessendorf::s_kDefaultTileLength);
    m.SetWindDirection(WSTessendorf::s_kDefaultWindDir);
    m.SetWindSpeed(WSTessendorf::s_kDefaultWindSpeed);
    m.SetAnimationPeriod(WSTessendorf::s_kDefaultAnimPeriod);
    m.SetPhillipsConst(WSTessendorf::s_kDefaultPhillipsConst);
    m.SetDamping(WSTessendorf::s_kDefaultPhillipsDamping);
    m.SetLambda(-1.0f);
    m.Prepare();
    float a = m.ComputeWaves(0.5f);
    const size_t dbytes = sizeof(WSTessendorf::Displacement) * m.GetDisplacementCount();
    const size_t nbytes = sizeof(WSTessendorf::Normal) * m.GetNormalCount();
    staging.resize(dbytes + nbytes);
    std::memcpy(staging.data(), m.GetDisplacements().data(), dbytes);
    std::memcpy(staging.data() + dbytes, m.GetNormals().data(), nbytes);
    auto w = m.GetWindDir();
    return a + m.GetTileSize() + m.GetTileLength() + w.x + w.y + m.GetWindSpeed() + m.GetAnimationPeriod() +
           m.GetPhillipsConst() + m.GetDamping() + m.GetDisplacementLambda() + m.GetMinHeight() + m.GetMaxHeight();
}
''')
    subprocess.check_call([GXX, "-std=c++17", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)])
    # with glm in scope the adaptor uses glm::vec2 / glm::vec4 like the reference.  glm is not a dependency of this
    # project, so a stand-in with glm's version macro and the members the caller and the adaptor touch takes its place.
    glm = tmp_path / "glm_standin"
    (glm / "glm").mkdir(parents=True)
    (glm / "glm" / "glm.hpp").write_text(r'''#pragma once
#define GLM_VERSION 999
namespace glm {
struct vec2 { float x, y; vec2(float x_ = 0.f, float y_ = 0.f) : x(x_), y(y_) {} };
struct vec4 { float x, y, z, w; vec4(float v = 0.f) : x(v), y(v), z(v), w(v) {} };
}
''')
    src2 = tmp_path / "iface_glm.cpp"
    src2.write_text('#include <glm/glm.hpp>\n' + src.read_text() +
                    '\nstatic_assert(std::is_same<WSTessendorf::Displacement, glm::vec4>::value, "glm types");\n'
                    'static_assert(std::is_same<decltype(std::declval<WSTessendorf&>().GetWindDir()), glm::vec2>::value,'
                    ' "glm wind");\n')
    subprocess.check_call([GXX, "-std=c++17", "-fsyntax-only", "-I", str(glm), "-I", os.path.join(ROOT, "include"),
                           str(src2)])


@pytest.mark.gpu
def test_frame_loop_matches_python_path():
    exe = _build_frame_loop()
    n, frames, seed = 256, 12, 4321
    out = subprocess.run([exe, str(n), str(frames), str(seed)], capture_output=True, text=True, check=True).stdout
    r = json.loads(out)
    import watersurfacerendering_b200 as W
    with W.WSTessendorf(n, 1000.0 * n / 512) as ws:
        ws.Prepare(seed=seed)
        t = np.float32(0.0)
        for _ in range(frames):
            t = np.float32(t + np.float32(np.float32(1.0 / 60.0) * np.float32(3.0)))
        a = ws.ComputeWaves(float(t))
        chk = float(ws.GetDisplacements().astype(np.float64).sum() + ws.GetNormals().astype(np.float64).sum())
        assert abs(r["t_last"] - float(t)) < 1e-6
        assert r["amplitude_last"] == pytest.approx(float(a), rel=1e-7)
        assert r["min_height"] == pytest.approx(float(ws.GetMinHeight()), rel=1e-7)
        assert r["checksum"] == pytest.approx(chk, rel=1e-9, abs=1e-3)
        assert r["tile_frames_per_s"] > 0
