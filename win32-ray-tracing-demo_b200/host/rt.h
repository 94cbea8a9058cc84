// rt.h -- host-side C++ API of the B200 ray tracer.
//
// It mirrors the platform-independent API of windy32/win32-ray-tracing-demo (src/RayTracingOpt):
// the same class names, constructor arguments and call sequence (build a GeometrySet of Plane /
// Sphere / Triangle / Tunnel geometries with SolidColor / Checker / RadianceChecker / Phong / Glass
// materials, a PerspectiveCamera, a RenderSetting, then call a RenderProc), so the reference's scene
// scripts read the same against it.  What differs is what happens behind the calls:
//   * geometries and materials carry parameters only; they are FLATTENED (flatten()) into the
//     SoA buffers of include/rtb.h and evaluated by the CUDA kernels -- there is no CPU shading or
//     intersection code in this library;
//   * Tunnel::init() runs the host builders (regular / flat grid, k-d median / SAH) and emits the
//     flattened accelerator directly (CSR cell directory, pre-order 8-byte k-d nodes);
//   * CudaRenderer::Render has the RenderProc signature and renders on the GPU through the C ABI;
//   * Geometry::intersect(Ray&) is served by a one-ray batch on the GPU.
// Reference citations are relative to src/RayTracingOpt/.
#ifndef RTB_HOST_RT_H
#define RTB_HOST_RT_H

#include <climits>
#include <cmath>
#include <cstdint>
#include <memory>
#include <string>
#include <vector>

#include "../../include/rtb.h"

namespace rt {

const float PI = 3.14159265359f; // Vector.h:8

// ---- math (Vector.h, Point.h, Color.h, Matrix.h) ----------------------------------------------
class Point;
class Vector
{
public:
    float x, y, z;
    Vector(float x = 0, float y = 0, float z = 0) : x(x), y(y), z(z) {}
    Vector(const Point &start, const Point &end);
    float length() const { return std::sqrt(x * x + y * y + z * z); }
    float sqrLength() const { return x * x + y * y + z * z; }
    float &operator[](int i) { return i == 0 ? x : (i == 1 ? y : z); }
    const float &operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
    Vector operator+(const Vector &b) const { return Vector(x + b.x, y + b.y, z + b.z); }
    Vector operator-(const Vector &b) const { return Vector(x - b.x, y - b.y, z - b.z); }
    Vector operator*(float b) const { return Vector(x * b, y * b, z * b); }
    Vector mult(const Vector &b) const { return Vector(x * b.x, y * b.y, z * b.z); }
    Vector &norm() { return *this = *this * (1 / std::sqrt(x * x + y * y + z * z)); }
    float dot(const Vector &b) const { return x * b.x + y * b.y + z * b.z; }
    float dot(const Point &p) const;
    Vector cross(const Vector &b) const { return Vector(y * b.z - z * b.y, z * b.x - x * b.z, x * b.y - y * b.x); }
    float angleTo(const Vector &b) const { return std::acos(dot(b) * (1.0f / (length() * b.length()))); }
};

class Point
{
public:
    float x, y, z;
    Point(float x = 0, float y = 0, float z = 0) : x(x), y(y), z(z) {}
    Point operator+(const Vector &v) const { return Point(x + v.x, y + v.y, z + v.z); }
    float &operator[](int i) { return i == 0 ? x : (i == 1 ? y : z); }
    const float &operator[](int i) const { return i == 0 ? x : (i == 1 ? y : z); }
};
inline Vector::Vector(const Point &s, const Point &e) : x(e.x - s.x), y(e.y - s.y), z(e.z - s.z) {}
inline float Vector::dot(const Point &p) const { return x * p.x + y * p.y + z * p.z; }

class Color
{
public:
    float r, g, b;
    Color() : r(0), g(0), b(0) {}
    Color(float r, float g, float b) : r(r), g(g), b(b) {}
    Color operator+(const Color &c) const { return Color(r + c.r, g + c.g, b + c.b); }
    Color operator*(float f) const { return Color(r * f, g * f, b * f); }
    Color mult(const Color &c) const { return Color(r * c.r, g * c.g, b * c.b); }
    void saturate() { r = r > 1.0f ? 1.0f : r; g = g > 1.0f ? 1.0f : g; b = b > 1.0f ? 1.0f : b; }
    static Color Red() { return Color(1, 0, 0); }
    static Color Green() { return Color(0, 1, 0); }
    static Color Blue() { return Color(0, 0, 1); }
    static Color Black() { return Color(0, 0, 0); }
    static Color White() { return Color(1, 1, 1); }
};

class Matrix
{
public:
    float m11, m12, m13, m21, m22, m23, m31, m32, m33;
    Matrix(float a, float b, float c, float d, float e, float f, float g, float h, float i)
        : m11(a), m12(b), m13(c), m21(d), m22(e), m23(f), m31(g), m32(h), m33(i) {}
    Point operator*(const Point &p) const
    {
        return Point(m11 * p.x + m12 * p.y + m13 * p.z, m21 * p.x + m22 * p.y + m23 * p.z, m31 * p.x + m32 * p.y + m33 * p.z);
    }
    Vector operator*(const Vector &p) const
    {
        return Vector(m11 * p.x + m12 * p.y + m13 * p.z, m21 * p.x + m22 * p.y + m23 * p.z, m31 * p.x + m32 * p.y + m33 * p.z);
    }
};

// ---- rays (Ray.h, RayContext.h, IntersectResult.h) --------------------------------------------
struct RayContext { bool inTunnel = false; int segment = -1; };
struct Ray
{
    Point origin;
    Vector direction;
    RayContext context;
    Ray(const Point &o, const Vector &d) : origin(o), direction(d) {}
    Point getPoint(float distance) const { return origin + direction * distance; }
};
class Geometry;
struct IntersectResult
{
    bool hit = false;
    Geometry *geometry = nullptr;
    float distance = 0;
    Point position;
    Vector normal;
    int id = -1; // flattened hit id (include/rtb.h convention)
    IntersectResult() {}
    IntersectResult(bool h) : hit(h) {}
};

// ---- materials (Material.h and subclasses) ----------------------------------------------------
class Material
{
public:
    float diffusiveness, reflectiveness, refractiveness;
    float refractive_index = 0;
    Material(float d, float r, float t) : diffusiveness(d), reflectiveness(r), refractiveness(t) {}
    virtual ~Material() {}
    void setRefractiveIndex(float index) { refractive_index = index; }
    virtual rtb_material flatten() const = 0; // replaces the CPU virtuals local()/emission()
protected:
    rtb_material base(int kind) const;
};
template <class T> using Ptr = std::shared_ptr<T>; // the reference's hand-rolled refcounted Ptr<T>

class SolidColorMaterial : public Material
{
public:
    Color localColor, emissionColor;
    SolidColorMaterial(const Color &local, const Color &emission, float d, float r, float t)
        : Material(d, r, t), localColor(local), emissionColor(emission) {}
    rtb_material flatten() const override;
};
class GlassMaterial : public SolidColorMaterial
{
public:
    GlassMaterial(float refractive_index = 1.46) : SolidColorMaterial(Color::White(), Color::Black(), 0, 0, 1)
    {
        setRefractiveIndex(refractive_index);
    }
};
class CheckerMaterial : public Material
{
public:
    enum checker_dir_t { xoz, xoy, yoz };
    float scale;
    checker_dir_t dir;
    CheckerMaterial(float scale, checker_dir_t dir = xoz, float reflectiveness = 0)
        : Material(1 - reflectiveness, reflectiveness, 0), scale(scale), dir(dir) {}
    rtb_material flatten() const override;
};
class RadianceCheckerMaterial : public Material
{
public:
    enum checker_dir_t { xoz, xoy, yoz };
    float radiance, scale;
    checker_dir_t dir;
    RadianceCheckerMaterial(float radiance, float scale, checker_dir_t dir = xoz)
        : Material(1, 0, 0), radiance(radiance), scale(scale), dir(dir) {}
    rtb_material flatten() const override;
};
class PhongMaterial : public Material
{
public:
    Color diffuse, specular;
    float shininess;
    PhongMaterial(const Color &diffuse, const Color &specular, float shininess, float reflectiveness = 0)
        : Material(1 - reflectiveness, reflectiveness, 0), diffuse(diffuse), specular(specular), shininess(shininess) {}
    rtb_material flatten() const override;
};

// ---- flattened scene owner --------------------------------------------------------------------
struct FlatScene
{
    std::vector<rtb_prim> prims;
    std::vector<rtb_material> materials;
    std::vector<const Material *> materialKeys; // de-duplication by object identity
    std::vector<float> looseTri;
    std::vector<float> tri;
    std::vector<int32_t> triMaterial;
    std::vector<rtb_cellword> gridWords;
    std::vector<uint32_t> gridCellStart, gridCellTris;
    std::vector<rtb_kdnode> kdNodes;
    std::vector<uint32_t> kdLeafTris;
    std::vector<float> cxFrames, cxEdges;  // convex accelerator (include/rtb.h: cx_*)
    std::vector<uint8_t> cxCellStatus;
    std::vector<int16_t> cxCellRange;
    std::vector<uint16_t> cxOrder;
    rtb_flat_scene view; // pointers into the vectors above; refreshed by finish()
    int nTop = 0;
    FlatScene();
    int materialIndex(const Material *m);
    void finish();
    size_t hostBytes() const;
};

// ---- geometries (Geometry.h, Plane.h, Sphere.h, Triangle.h, GeometrySet.h) --------------------
class Geometry
{
public:
    Ptr<Material> material;
    Geometry() {}
    virtual ~Geometry() {}
    // Reference Geometry.h:17.  Served by the GPU: the geometry is flattened into a one-object
    // device scene (cached) and a one-ray batch goes through rtb_intersect_rays.
    virtual IntersectResult intersect(Ray &ray);
    void setMaterial(const Ptr<Material> &m) { material = m; }
    virtual void flatten(FlatScene &out) const = 0;
    virtual void invalidate();
    // number of top-level hit ids the geometry takes (GeometrySet::resolveHit): one, a mesh one per triangle
    virtual int topLevelIds() const { return 1; }
    // true: topLevelIds() may differ from 1 (and change as the geometry grows)
    virtual bool variableIds() const { return false; }
private:
    struct DeviceCache;
    std::shared_ptr<DeviceCache> cache_;
protected:
    virtual Geometry *resolveHit(int id);
};

class Plane : public Geometry
{
    Vector normal;
    Point position;
    float dist;
public:
    Plane(const Vector &normal, float dist) : normal(normal), dist(dist) { position = Point(0, 0, 0) + normal * dist; }
    void flatten(FlatScene &out) const override;
};

class Sphere : public Geometry
{
    Point center;
    float radius;
public:
    Sphere(const Point &center, float radius) : center(center), radius(radius) {}
    void flatten(FlatScene &out) const override;
};

class Triangle : public Geometry
{
public:
    Point a, b, c;
    Vector normal;
    Triangle() {}
    Triangle(const Point &a, const Point &b, const Point &c, const Vector &normal) : a(a), b(b), c(c), normal(normal) {}
    Triangle(const Point &a, const Point &b, const Point &c) : a(a), b(b), c(c)
    {
        normal = Vector(a, b).cross(Vector(b, c)).norm();
    }
    void getBoundingBox(Point &min, Point &max) const;
    void flatten(FlatScene &out) const override;
};

// A triangle mesh: one RTB_PRIM_MESH record, traversed on the device through a hierarchy built at upload.  It hits what the
// same triangles added one by one (GeometrySet::addStlFile) hit, with the same ids: triangle k of the mesh is top-level id
// base + k (include/rtb.h: RTB_PRIM_MESH).  No reference counterpart: the reference loads every facet as a loose Triangle.
class TriangleMesh : public Geometry
{
    std::vector<float> tris; // [n][12]: a, b, c, normal, as the loose_tri records of include/rtb.h
public:
    size_t count() const { return tris.size() / 12; }
    void add(const Point &a, const Point &b, const Point &c, const Vector &normal); // drops the cached device upload
    void flatten(FlatScene &out) const override;
    int topLevelIds() const override { return (int)count(); }
    bool variableIds() const override { return true; }
protected:
    Geometry *resolveHit(int id) override;
};

class GeometrySet : public Geometry
{
    std::vector<Geometry *> geometries;
    bool variableIds_ = false; // some geometry may take more or less than one hit id: resolveHit walks the list
public:
    void add(Geometry *geometry) { geometries.push_back(geometry); variableIds_ = variableIds_ || geometry->variableIds(); invalidate(); }
    Geometry *last() { return geometries.empty() ? nullptr : geometries.back(); }
    size_t size() const { return geometries.size(); }
    bool addStlFile(const char *filename, Ptr<Material> material);
    bool addStlFile(const char *filename, Ptr<Material> material, const Matrix &matrix, const Vector &offset);
    // the same facets as ONE TriangleMesh (same loose_tri records, same hit ids)
    bool addStlMesh(const char *filename, Ptr<Material> material);
    bool addStlMesh(const char *filename, Ptr<Material> material, const Matrix &matrix, const Vector &offset);
    void clear();
    void flatten(FlatScene &out) const override;
    // batch form of intersect(): n rays [n][6] -> results (GPU)
    bool intersectBatch(const float *rays, int64_t n, int32_t *hitId, float *hitT, float *position, float *normal);
    ~GeometrySet() override;
protected:
    Geometry *resolveHit(int id) override;
};

// ---- tunnel (Tunnel.h, TunnelGenerator.h, PerformanceTest/Accelerator.h) ----------------------
struct TunnelTriangle { Point a, b, c; Vector normal; int material; }; // material: 0 wall, 1 ground

class Tunnel : public Geometry
{
public:
    enum Algorithm { Linear = 0, RegularGrid = 1, FlatGrid = 2, KdTreeStandard = 3, KdTreeSAH = 4, Convex = 5, ConvexSimple = 6 };
    Algorithm algorithm = Linear;
    float height = 0, width = 0;
    std::vector<Point> path;
    std::vector<Point> crossSection;                  // the polygon at the origin, Tunnel.h:11
    std::vector<Vector> ringNormals;                  // PerformanceTest/Tunnel.h:16 `nvs` (that program's generator only)
    std::vector<std::vector<TunnelTriangle>> surface; // [segment][j], reference Tunnel.h:13
    Ptr<Material> groundMaterial, wallMaterial;

    // builder parameters; defaults are the reference's compile-time constants
    int gridResolution = 400; // Tunnel.cpp:381,395-404
    int kdLeafSize = 8;       // Tunnel.cpp:550
    int kdMaxDepth = 18;
    int sahCandidates = 100;  // Tunnel.cpp:679
    // KdTreeSAH builds with PerformanceTest's builder (KdTreeAcc.cpp: event-sweep SAH + automatic termination)
    // instead of RayTracingOpt's 99-candidate one; set by TunnelGenerator::performanceTestVariant
    bool performanceTestBuilders = false;
    // RegularGrid / FlatGrid: leave the grid to the device builder (rtb_scene_upload, include/rtb.h:
    // grid_build_resolution) instead of building it here; init() then only records the request.  The default for
    // newly generated tunnels is Tunnel::gridOnDeviceDefault (false: host build, needed for host-side statistics).
    bool gridOnDevice = false;
    static bool gridOnDeviceDefault;
    // RegularGrid / FlatGrid: a triangle enters a cell only if it passes the exact overlap test Triangle::intersectWithGrid
    // (reference Triangle.cpp:152-199), the alternative the reference keeps compiled out at Tunnel.cpp:435-445; default
    // false = the bounding-box binning the reference ships.  Host and device builders honour it (csrc/rtb_sat.h).
    bool exactGridBinning = false;
    static bool exactGridBinningDefault;
    // KdTreeSAH: leave the tree to the device builder (rtb_scene_upload, include/rtb.h: kd_build_*; csrc/rtb_build_kd.cuh)
    // instead of building it here; init() then only records the request (RayTracingOpt's 99-candidate builder only).
    bool kdOnDevice = false;
    static bool kdOnDeviceDefault;

    // Reference Tunnel.cpp:116-133: builds the accelerator selected by `algorithm`.
    void init();
    void flatten(FlatScene &out) const override;
    size_t triangleCount() const;

    struct BuildStats
    {
        int gridX = 0, gridY = 0, gridZ = 0;
        int64_t cellsNonEmpty = 0, cellEntries = 0, cellMax = 0;
        int64_t kdNodes = 0, kdLeaves = 0, kdLeafRefs = 0, kdMaxDepth = 0;
    } stats;

private:
    friend class TunnelGenerator;
    bool built_ = false;
    // flattened accelerator (what the builders emit)
    float gridOrigin_[3] = {0, 0, 0}, gridCell_[3] = {0, 0, 0};
    int gridDims_[3] = {0, 0, 0};
    std::vector<rtb_cellword> gridWords_;
    std::vector<uint32_t> gridCellStart_, gridCellTris_;
    float kdMin_[3] = {0, 0, 0}, kdMax_[3] = {0, 0, 0};
    std::vector<rtb_kdnode> kdNodes_;
    std::vector<uint32_t> kdLeafTris_;
    std::vector<float> cxFrames_, cxEdges_;
    std::vector<uint8_t> cxCellStatus_;
    std::vector<int16_t> cxCellRange_;
    std::vector<uint16_t> cxOrder_;
    int cxTable_ = 0;
    void initConvex();
    void collect(std::vector<TunnelTriangle> &flat) const;
    void initGrid(const std::vector<TunnelTriangle> &tris);
    void initKdTree(const std::vector<TunnelTriangle> &tris);
};

class TunnelGenerator
{
public:
    // false: RayTracingOpt's generator (rings turned by their segment's direction, TunnelGenerator.cpp:262-290);
    // true:  PerformanceTest's (rings turned by the averaged directions of the adjoining segments,
    //        src/PerformanceTest/TunnelGenerator.cpp:243-279) and its k-d builder -- the two programs differ there
    bool performanceTestVariant = false;
    // Reference TunnelGenerator.cpp:197-366.
    bool create(float rectWidth, float rectHeight, float archHeight, float pathRadius, float pathAngle,
                int archSegments, int pathSegments, GeometrySet &scene, Ptr<Material> groundMaterial,
                Ptr<Material> wallMaterial, Tunnel::Algorithm algorithm);
};

// PerformanceTest/Accelerator.h:6-15 -- the per-ray plugin interface, kept for callers that
// drive a tunnel directly; init() = Tunnel::init(), intersect() = GPU one-ray batch.
class Accelerator
{
public:
    Tunnel *tunnel;
    explicit Accelerator(Tunnel *t) : tunnel(t) {}
    virtual ~Accelerator() {}
    virtual void init() { tunnel->init(); }
    virtual IntersectResult intersect(Ray &ray) { return tunnel->intersect(ray); }
};

// ---- camera, settings (Camera.h, RenderSetting.h) ---------------------------------------------
class PerspectiveCamera
{
    Point eye;
    Vector front, up, right;
    float ratio, xcenter, fov, fovScale, forward;
public:
    PerspectiveCamera(const Point &eye, Vector front, const Vector &up, float ratio, float fov, float forward = 0.0f);
    Ray generateRay(float x, float y) const; // Camera.cpp:20-26 (host convenience; kernels generate their own)
    rtb_camera flatten() const;
};

struct RenderSetting
{
    bool enableMonteCarlo;
    int maxDepth, terminationDepth, singleTracingDepth;
    static RenderSetting HighSpeed() { return {true, 6, 2, 0}; }
    static RenderSetting HighQuality() { return {true, 8, INT_MAX, INT_MAX}; }
    static RenderSetting Default() { return {true, INT_MAX, 5, 2}; }
    static RenderSetting Simple() { return {false, 20, INT_MAX, 0}; }
    rtb_render_setting flatten() const { return {enableMonteCarlo ? 1 : 0, maxDepth, terminationDepth, singleTracingDepth}; }
};

// ---- PerformanceTest (src/PerformanceTest): its camera and its benchmark, GPU-served -------------------
class Camera
{ // PerformanceTest/Camera.h:7-20 -- fixed 1.274 x 1.0 image plane, no fov / ratio / forward
    Point eye;
    Vector front, up, right;
public:
    Camera(const Point &eye, Vector front, const Vector &up);
    Ray generateRay(float x, float y) const;
};

struct PerformanceTest
{ // PerformanceTest/main.cpp: tunnel + exit plane, N rays bounced to the exit (<= 200 reflections)
    GeometrySet scene;
    Tunnel *tunnel = nullptr;
    double buildMs = 0, preprocessMs = 0;
    bool build(float pathRadius, float pathAngle, int archSeg, int pathSeg, Tunnel::Algorithm algorithm); // main.cpp:61-81,134-140
    static Tunnel *buildScene(GeometrySet &scene, float pathRadius, float pathAngle, int archSeg, int pathSeg,
                              Tunnel::Algorithm algorithm); // the scene alone, accelerator not yet built
    // xy: n camera samples in [0,1]^2 (the reference draws them with rand()); returns the trace kernel's ms, < 0 on error
    double run(const float *xy, int n, int maxDepth, int32_t *reached, int32_t *depth, int32_t *lastId, float *lastPos,
               int64_t *totalRays);
};

// ---- render entry point and scene scripts (Scripts.h) -----------------------------------------
typedef void (*LogCallback)(const char *str);
typedef void (*ProgressCallback)(int cur, int total);
typedef int (*RenderProc)(GeometrySet &scene, PerspectiveCamera &camera, RenderSetting &setting, ProgressCallback progress);

class Script
{
public:
    enum { FLAG_TUNNEL = 0x1, FLAG_MONTE_CARLO = 0x2 };
    const char *name;
    int flags;
    int tunnelSegments; // valid when FLAG_TUNNEL
    int samples;        // valid when FLAG_MONTE_CARLO
    int preset;         // 1..5
    std::string stlPath = "ball.stl";
    static bool stlAsMeshDefault; // preset 3 loads its STL with addStlMesh instead of addStlFile
    Script(const char *name, int flags, int tunnelSegments, int samples, int preset)
        : name(name), flags(flags), tunnelSegments(tunnelSegments), samples(samples), preset(preset) {}
    virtual ~Script() {}
    // Reference Scripts.h:38-39.
    virtual void Run(RenderProc render, int tunnelAlgorithm, LogCallback log, ProgressCallback progress,
                     int &prepareTime, int &execTime);
    // Builds the preset's scene / camera / setting (Scripts.cpp:22-278) without rendering.
    bool Build(GeometrySet &scene, std::unique_ptr<PerspectiveCamera> &camera, RenderSetting &setting,
               int tunnelAlgorithm, int &prepareTime) const;
};
extern Script *scripts[5];

// The GPU RenderProc.  `Render` has the reference's RenderProc signature (Scripts.h:11-12); image
// size and sample count are object state because the reference keeps them in file statics
// (MainWindow.cpp:33-36).  Returns elapsed render milliseconds, negative on error (message through
// lastError()).
class CudaRenderer
{
public:
    static CudaRenderer &instance();
    void configure(int width, int height, int samples, int device = 0, uint64_t seed = 0);
    // Render on `n` devices (0 .. n - 1) driven by this one host thread: the frame is sharded over them and every
    // device stores its tiles straight into the one host frame (rtb_multi_render).  1 = the single device given to
    // configure().  SURVEY 8b threading row.
    void setDevices(int n);
    int devices() const { return nDevices_; }
    // The reference's Render has no error channel (Scripts.h:11-12): failures are reported through this callback (the
    // LogCallback the caller also hands to Script::Run) and surface as a negative return value.
    void setLog(LogCallback log) { log_ = log; }
    static int Render(GeometrySet &scene, PerspectiveCamera &camera, RenderSetting &setting, ProgressCallback progress);
    const std::vector<float> &image() const { return image_; } // reference order: index = x*height + y
    // Output stage of the reference's Render (MainWindow.cpp:305-311): when enabled the GPU saturates and
    // quantises, only 3 bytes per pixel come back, and pixels() holds R,G,B in the same x*height + y order.
    void setOutput8bit(bool on) { output8_ = on; }
    const std::vector<unsigned char> &pixels() const { return pixels_; }
    // 24-bit BMP of pixels() (the reference's Save-As path: MainWindow.cpp:664-708 + Utils.cpp:78-119;
    // rows bottom-up, B,G,R; unlike the reference rows are padded to 4 bytes and biPlanes is 1, so the
    // file is valid for every width).
    bool saveBitmap(const char *filename) const;
    const rtb_stats &stats() const { return stats_; }
    const std::string &lastError() const { return error_; }
    rtb_ctx *context();
    void shutdown();
    int width() const { return width_; }
    int height() const { return height_; }
private:
    int failed(int code, const char *what, const char *detail);
    rtb_multi *multi();
    int width_ = 400, height_ = 300, samples_ = 1, device_ = 0, nDevices_ = 1;
    uint64_t seed_ = 0;
    rtb_ctx *ctx_ = nullptr;
    rtb_multi *multi_ = nullptr;
    LogCallback log_ = nullptr;
    std::vector<float> image_;
    std::vector<unsigned char> pixels_;
    bool output8_ = false;
    float *pinned_ = nullptr;
    size_t pinnedFloats_ = 0;
    rtb_stats stats_;
    std::string error_;
};

} // namespace rt
#endif
