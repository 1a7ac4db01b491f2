// wso_tessendorf_adaptor.hpp — header-only C++ host side of the drop-in boundary.
//
// Re-exposes, on top of the C ABI in wsocean.h, exactly the public interface of the reference's
// `class WSTessendorf` (reference: src/scene/WSTessendorf.h:58-122) so that its only caller,
// src/scene/WaterSurfaceMesh.cpp (Prepare at :127/:898, ComputeWaves at :131/:151, getters at :172-179,
// map reads at :705-741, setters at :880-902), compiles unchanged when
//     src/scene/WSTessendorf.h   is replaced by   #include <wso_tessendorf_adaptor.hpp>
// and src/scene/WSTessendorf.cpp + FFTW are dropped from the build (see INTEGRATION.md).
//
// Differences a caller can observe:
//   * none in the signatures: GetDisplacements()/GetNormals() return const std::vector<vec4>& exactly as
//     WSTessendorf.h:95-101 does.  The vectors are owned here, sized and filled with the reference's defaults in
//     Prepare() (WSTessendorf.cpp:48-54), page-locked in place (wso_register_host) and written by the device-to-host
//     copies of every ComputeWaves() - the memcpy in WaterSurfaceMesh::CopyModelTessDataToStagingBuffer
//     (WaterSurfaceMesh.cpp:701-755) reads them as before;
//   * errors of the CUDA path throw std::runtime_error (the reference has no failure modes besides asserts).
// glm is used when the including translation unit has already included <glm/glm.hpp> (as the reference's
// pch.h does); otherwise two minimal POD vectors stand in so the header is self-contained.
#ifndef WSO_TESSENDORF_ADAPTOR_HPP_
#define WSO_TESSENDORF_ADAPTOR_HPP_

#include <cstddef>
#include <cstdint>
#include <stdexcept>
#include <string>
#include <vector>

#include "wsocean.h"

#if defined(GLM_VERSION) || defined(GLM_SETUP_INCLUDED)
namespace wso_adaptor {
using vec2 = glm::vec2;
using vec4 = glm::vec4;
}  // namespace wso_adaptor
#else
namespace wso_adaptor {
struct vec2 {
    float x, y;
    vec2(float x_ = 0.0f, float y_ = 0.0f) : x(x_), y(y_) {}
};
struct alignas(16) vec4 {
    float x, y, z, w;
};
}  // namespace wso_adaptor
#endif

class WSTessendorf {
public:
    static constexpr uint32_t s_kDefaultTileSize{512};
    static constexpr float s_kDefaultTileLength{1000.0f};
    static inline const wso_adaptor::vec2 s_kDefaultWindDir{1.0f, 1.0f};
    static constexpr float s_kDefaultWindSpeed{30.0f};
    static constexpr float s_kDefaultAnimPeriod{200.0f};
    static constexpr float s_kDefaultPhillipsConst{3e-7f};
    static constexpr float s_kDefaultPhillipsDamping{0.1f};

    using Displacement = wso_adaptor::vec4;  // RGBA32F texel (VK_FORMAT_R32G32B32A32_SFLOAT)
    using Normal = wso_adaptor::vec4;

    explicit WSTessendorf(uint32_t tileSize = s_kDefaultTileSize, float tileLength = s_kDefaultTileLength,
                          int cudaDevice = 0) {
        wso_params p;
        wso_default_params(&p);
        // like the reference constructor, a non power-of-two size is ignored (WSTessendorf.cpp:459-468)
        if (tileSize != 0 && (tileSize & (tileSize - 1)) == 0) p.tile_size = tileSize;
        p.tile_length = tileLength;
        Check(wso_create(&p, cudaDevice, 1, 1, &m_Ctx), "wso_create");
    }
    ~WSTessendorf() {
        ReleaseMaps();
        wso_destroy(m_Ctx);
    }
    WSTessendorf(const WSTessendorf&) = delete;
    WSTessendorf& operator=(const WSTessendorf&) = delete;

    void Prepare() {
        Check(wso_prepare(m_Ctx, 0, /*reseed=*/0, 0), "wso_prepare");
        ResizeMaps();
    }

    float ComputeWaves(float time) {
        float amplitude = 0.0f;
        Check(wso_compute_to_host(m_Ctx, 1, nullptr, &time, reinterpret_cast<float*>(m_Displacements.data()),
                                  reinterpret_cast<float*>(m_Normals.data()), &amplitude, &m_MinHeight, &m_MaxHeight),
              "wso_compute_to_host");
        return amplitude;
    }

    // ---- getters (reference: WSTessendorf.h:82-101)
    auto GetTileSize() const { return Params().tile_size; }
    auto GetTileLength() const { return Params().tile_length; }
    auto GetWindDir() const {
        const wso_params p = Params();
        return wso_adaptor::vec2(p.wind_dir_x, p.wind_dir_y);
    }
    auto GetWindSpeed() const { return Params().wind_speed; }
    auto GetAnimationPeriod() const { return Params().anim_period; }
    auto GetPhillipsConst() const { return Params().phillips_const; }
    auto GetDamping() const { return Params().damping; }
    auto GetDisplacementLambda() const { return Params().lambda; }
    float GetMinHeight() const { return m_MinHeight; }
    float GetMaxHeight() const { return m_MaxHeight; }

    size_t GetDisplacementCount() const { return m_Displacements.size(); }
    const std::vector<Displacement>& GetDisplacements() const { return m_Displacements; }
    size_t GetNormalCount() const { return m_Normals.size(); }
    const std::vector<Normal>& GetNormals() const { return m_Normals; }

    // ---- setters (reference: WSTessendorf.cpp:459-505)
    void SetTileSize(uint32_t size) {
        wso_params p = Params();
        p.tile_size = size;
        const int rc = wso_set_params(m_Ctx, 0, &p);
        if (rc != WSO_OK && rc != WSO_ERR_BAD_TILE_SIZE) Check(rc, "wso_set_params");
    }
    void SetTileLength(float length) { Set([&](wso_params& p) { p.tile_length = length; }); }
    void SetWindDirection(const wso_adaptor::vec2& w) {
        Set([&](wso_params& p) { p.wind_dir_x = w.x; p.wind_dir_y = w.y; });
    }
    void SetWindSpeed(float v) { Set([&](wso_params& p) { p.wind_speed = v; }); }
    void SetAnimationPeriod(float T) { Set([&](wso_params& p) { p.anim_period = T; }); }
    void SetPhillipsConst(float A) { Set([&](wso_params& p) { p.phillips_const = A; }); }
    void SetLambda(float lambda) { Check(wso_set_lambda(m_Ctx, 0, lambda), "wso_set_lambda"); }
    // Extension (not in the reference class): its compile-time COMPUTE_JACOBIAN switch (WSTessendorf.cpp:421-428, dead
    // code there) at run time - displacement.w = Jacobian of the horizontal displacement instead of 1.
    void SetComputeJacobian(bool on) { Check(wso_set_compute_jacobian(m_Ctx, on ? 1 : 0), "wso_set_compute_jacobian"); }
    void SetDamping(float damping) { Set([&](wso_params& p) { p.damping = damping; }); }
    // Extension (not in the reference class): the surface above n world points xz[2i], xz[2i+1] (host arrays) - height,
    // normal and undisplaced origin - sampled from the maps of the last ComputeWaves() (slot 0), with `iterations`
    // fixed-point steps of the choppy-displacement inversion (wsocean.h, "Surface queries").  Blocking.
    void QuerySurface(const float* xz, uint32_t n, wso_surface_sample* out, uint32_t iterations = 4) {
        const uint32_t slot = 0;
        Check(wso_query_surface_host(m_Ctx, 1, &slot, iterations, n, xz, out), "wso_query_surface_host");
    }
    // Extension: the first point at or under the surface of slot 0 along n rays, rays[8i..8i+7] = (ox, oy, oz, tmax,
    // dx, dy, dz, unused) (host arrays), marched and refined as `p` says (wsocean.h, "Ray casts").  Blocking.
    void RaycastSurface(const float* rays, uint32_t n, wso_ray_hit* out, const wso_ray_params& p) {
        const uint32_t slot = 0;
        Check(wso_raycast_surface_host(m_Ctx, 1, &slot, &p, n, rays, out), "wso_raycast_surface_host");
    }

    // ---- extensions: device pointers for zero-copy consumers (e.g. Vulkan external memory, row f-2)
    void* GetDisplacementsDevice() const { return DevicePtr(WSO_MAP_DISPLACEMENT); }
    void* GetNormalsDevice() const { return DevicePtr(WSO_MAP_NORMAL); }
    wso_ctx* Handle() const { return m_Ctx; }

private:
    wso_params Params() const {
        wso_params p;
        Check(wso_get_params(m_Ctx, 0, &p), "wso_get_params");
        return p;
    }
    template <typename F>
    void Set(F&& f) {
        wso_params p = Params();
        f(p);
        Check(wso_set_params(m_Ctx, 0, &p), "wso_set_params");
    }
    // reference: Prepare() resizes both maps to N*N texels with default contents (WSTessendorf.cpp:48-54); a resize keeps
    // what is already there, like std::vector::resize does in the reference
    void ResizeMaps() {
        const size_t n = (size_t)GetTileSize() * GetTileSize();
        if (m_Displacements.size() == n && m_Normals.size() == n && m_Registered) return;
        ReleaseMaps();
        Displacement d0;
        d0.x = d0.y = d0.z = d0.w = 0.0f;
        Normal n0;
        n0.x = 0.0f; n0.y = 1.0f; n0.z = 0.0f; n0.w = 0.0f;
        m_Displacements.resize(n, d0);
        m_Normals.resize(n, n0);
        // page-lock the vectors' storage where it lies: the device-to-host copies then run at full PCIe speed
        m_Registered = wso_register_host(m_Displacements.data(), n * sizeof(Displacement)) == WSO_OK;
        if (m_Registered && wso_register_host(m_Normals.data(), n * sizeof(Normal)) != WSO_OK) {
            wso_unregister_host(m_Displacements.data());
            m_Registered = false;
        }
    }
    void ReleaseMaps() {
        if (m_Registered) {
            wso_unregister_host(m_Displacements.data());
            wso_unregister_host(m_Normals.data());
            m_Registered = false;
        }
    }
    void* DevicePtr(int which) const {
        void* p = nullptr;
        Check(wso_map_device(m_Ctx, which, 0, &p, nullptr), "wso_map_device");
        return p;
    }
    void Check(int rc, const char* what) const {
        if (rc != WSO_OK)
            throw std::runtime_error(std::string(what) + " failed (" + std::to_string(rc) +
                                     "): " + wso_last_error(m_Ctx));
    }

    wso_ctx* m_Ctx{nullptr};
    std::vector<Displacement> m_Displacements;
    std::vector<Normal> m_Normals;
    bool m_Registered{false};
    float m_MinHeight{-1.0f};  // reference: WSTessendorf.h:226-227
    float m_MaxHeight{1.0f};
};

#endif  // WSO_TESSENDORF_ADAPTOR_HPP_
