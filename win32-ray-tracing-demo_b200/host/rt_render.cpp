// rt_render.cpp -- the GPU RenderProc (CudaRenderer), the preset scene scripts, the GPU-served
// Geometry::intersect, and a small C API (rtbh_*) used by the Python tests / bench to reach the
// host builders and the drop-in entry point.
#include "rt.h"

#include <chrono>
#include <cstdio>
#include <cstring>
#include <mutex>

namespace rt {

static double nowMs()
{
    return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ---- CudaRenderer -------------------------------------------------------------------------------
CudaRenderer &CudaRenderer::instance()
{
    static CudaRenderer r;
    return r;
}

void CudaRenderer::configure(int width, int height, int samples, int device, uint64_t seed)
{
    if (ctx_ && device != device_) shutdown();
    width_ = width; height_ = height; samples_ = samples; device_ = device; seed_ = seed;
}

void CudaRenderer::setDevices(int n)
{
    if (n < 1) n = 1;
    if (n != nDevices_ && multi_) { rtb_multi_shutdown(multi_); multi_ = nullptr; }
    nDevices_ = n;
}

rtb_ctx *CudaRenderer::context()
{
    if (!ctx_)
    {
        const int rc = rtb_init(device_, &ctx_);
        if (rc != RTB_OK) { error_ = rtb_last_error(nullptr); ctx_ = nullptr; }
    }
    return ctx_;
}

rtb_multi *CudaRenderer::multi()
{
    if (!multi_)
    {
        const int rc = rtb_multi_init(nDevices_, nullptr, &multi_);
        if (rc != RTB_OK) { error_ = rtb_last_error(nullptr); multi_ = nullptr; }
    }
    return multi_;
}

void CudaRenderer::shutdown()
{
    if (pinned_) rtb_host_free(pinned_);
    pinned_ = nullptr;
    pinnedFloats_ = 0;
    if (ctx_) rtb_shutdown(ctx_);
    ctx_ = nullptr;
    if (multi_) rtb_multi_shutdown(multi_);
    multi_ = nullptr;
}

int CudaRenderer::failed(int code, const char *what, const char *detail)
{
    error_ = std::string(what) + ": " + (detail ? detail : "");
    if (log_) log_(("CudaRenderer: " + error_ + "\r\n").c_str()); // the reference's log lines end in \r\n (Scripts.cpp)
    return code;
}

// rtb_progress_fn -> ProgressCallback(cur, total) in the reference's unit, image rows (MainWindow.cpp:271)
struct ProgressAdapter { ProgressCallback fn; int height; int last; };
static void progressTrampoline(int64_t done, int64_t total, void *user)
{
    ProgressAdapter *a = static_cast<ProgressAdapter *>(user);
    const int cur = total > 0 ? (int)((done * a->height) / total) : a->height;
    if (cur != a->last) { a->last = cur; a->fn(cur, a->height); }
}

int CudaRenderer::Render(GeometrySet &scene, PerspectiveCamera &camera, RenderSetting &setting, ProgressCallback progress)
{ // replaces reference MainWindow.cpp:251-316
    CudaRenderer &self = instance();
    const bool many = self.nDevices_ > 1;
    rtb_ctx *ctx = many ? nullptr : self.context();
    rtb_multi *mul = many ? self.multi() : nullptr;
    if (!ctx && !mul) return self.failed(-1, "no CUDA device", self.error_.c_str());
    const double t0 = nowMs();
    FlatScene flat;
    scene.flatten(flat);
    flat.finish();
    rtb_scene *dev = nullptr;
    rtb_multi_scene *mdev = nullptr;
    int rc = many ? rtb_multi_scene_upload(mul, &flat.view, &mdev) : rtb_scene_upload(ctx, &flat.view, &dev);
    if (rc != RTB_OK) return self.failed(-2, "scene upload", many ? rtb_multi_last_error(mul) : rtb_last_error(ctx));
    auto release = [&]() { if (many) rtb_multi_scene_free(mul, mdev); else rtb_scene_free(ctx, dev); };
    const rtb_camera cam = camera.flatten();
    const rtb_render_setting rs = setting.flatten();
    rtb_frame frame;
    memset(&frame, 0, sizeof(frame));
    frame.width = self.width_; frame.height = self.height_; frame.samples = self.samples_;
    frame.seed = self.seed_; frame.rank = 0; frame.world = 1; frame.row_block = 8;
    frame.layout = RTB_LAYOUT_REFERENCE | (self.output8_ ? RTB_OUTPUT_RGB8 : 0); // colors[x*height + y], MainWindow.cpp:276
    const size_t floats = (size_t)self.width_ * self.height_ * 3;
    if (floats > self.pinnedFloats_)
    { // page-locked frame: the devices store their pixels straight into it
        if (self.pinned_) rtb_host_free(self.pinned_);
        self.pinned_ = nullptr;
        self.pinnedFloats_ = 0;
        void *p = nullptr;
        if (rtb_host_alloc(floats * sizeof(float), &p) != RTB_OK) { release(); return self.failed(-4, "rtb_host_alloc", rtb_last_error(nullptr)); }
        self.pinned_ = (float *)p;
        self.pinnedFloats_ = floats;
    }
    ProgressAdapter adapter = {progress, self.height_, -1};
    if (many) rtb_multi_set_progress(mul, progress ? progressTrampoline : nullptr, &adapter);
    else rtb_set_progress(ctx, progress ? progressTrampoline : nullptr, &adapter);
    rc = many ? rtb_multi_render(mul, mdev, &cam, &rs, &frame, self.pinned_, &self.stats_)
              : rtb_render(ctx, dev, &cam, &rs, &frame, self.pinned_, &self.stats_);
    if (many) rtb_multi_set_progress(mul, nullptr, nullptr);
    else rtb_set_progress(ctx, nullptr, nullptr);
    release();
    if (rc != RTB_OK) return self.failed(-3, "render", many ? rtb_multi_last_error(mul) : rtb_last_error(ctx));
    if (self.output8_)
    {
        const unsigned char *bytes = reinterpret_cast<const unsigned char *>(self.pinned_);
        self.pixels_.assign(bytes, bytes + floats);
        self.image_.clear();
    }
    else
    {
        self.image_.assign(self.pinned_, self.pinned_ + floats);
        self.pixels_.clear();
    }
    if (progress && adapter.last != self.height_) progress(self.height_, self.height_);
    const double ms = nowMs() - t0;
    return ms < 1.0 ? 1 : (int)(ms + 0.5);
}

bool CudaRenderer::saveBitmap(const char *filename) const
{
    if (pixels_.size() != (size_t)width_ * height_ * 3) return false;
    const uint32_t rowBytes = ((uint32_t)width_ * 3 + 3) & ~3u, size = rowBytes * (uint32_t)height_;
    unsigned char header[54];
    memset(header, 0, sizeof(header));
    auto put32 = [&](int at, uint32_t v) { memcpy(header + at, &v, 4); };
    auto put16 = [&](int at, uint16_t v) { memcpy(header + at, &v, 2); };
    put16(0, 0x4D42); put32(2, 54 + size); put32(10, 54);                  // BITMAPFILEHEADER
    put32(14, 40); put32(18, (uint32_t)width_); put32(22, (uint32_t)height_); // BITMAPINFOHEADER
    put16(26, 1); put16(28, 24); put32(34, size);
    FILE *fp = fopen(filename, "wb");
    if (!fp) return false;
    std::vector<unsigned char> row(rowBytes, 0);
    bool ok = fwrite(header, 1, sizeof(header), fp) == sizeof(header);
    for (int y = height_ - 1; y >= 0 && ok; y--)
    { // bottom-up rows, B G R (MainWindow.cpp:672-680)
        for (int x = 0; x < width_; x++)
        {
            const unsigned char *p = &pixels_[3 * ((size_t)x * height_ + y)];
            row[3 * x] = p[2]; row[3 * x + 1] = p[1]; row[3 * x + 2] = p[0];
        }
        ok = fwrite(row.data(), 1, rowBytes, fp) == rowBytes;
    }
    fclose(fp);
    return ok;
}

// ---- GPU-served single-ray queries --------------------------------------------------------------
struct Geometry::DeviceCache
{
    rtb_scene *scene = nullptr;
    ~DeviceCache()
    {
        if (scene) rtb_scene_free(CudaRenderer::instance().context(), scene);
    }
};

void Geometry::invalidate() { cache_.reset(); }
Geometry *Geometry::resolveHit(int) { return this; }

Geometry *TriangleMesh::resolveHit(int) { return this; }

Geometry *GeometrySet::resolveHit(int id)
{
    if (!variableIds_)
    { // one id per geometry
        if (id >= 0 && id < (int)geometries.size()) return geometries[id];
        return geometries.empty() ? this : geometries.back(); // tunnel triangle ids follow the top-level ones
    }
    int base = 0; // a mesh takes one id per triangle
    for (Geometry *g : geometries)
    {
        const int n = g->topLevelIds();
        if (id >= base && id < base + n) return g;
        base += n;
    }
    return geometries.empty() ? this : geometries.back(); // tunnel triangle ids follow the top-level ones
}

static rtb_scene *uploadGeometry(const Geometry &g)
{
    rtb_ctx *ctx = CudaRenderer::instance().context();
    if (!ctx) return nullptr;
    FlatScene flat;
    g.flatten(flat);
    flat.finish();
    rtb_scene *dev = nullptr;
    if (rtb_scene_upload(ctx, &flat.view, &dev) != RTB_OK) return nullptr;
    return dev;
}

IntersectResult Geometry::intersect(Ray &ray)
{
    IntersectResult res(false);
    if (!cache_)
    {
        cache_ = std::make_shared<DeviceCache>();
        cache_->scene = uploadGeometry(*this);
    }
    if (!cache_->scene) return res;
    const float r[6] = {ray.origin.x, ray.origin.y, ray.origin.z, ray.direction.x, ray.direction.y, ray.direction.z};
    int32_t id = -1;
    float t = 0, pos[3], nrm[3];
    if (rtb_intersect_rays(CudaRenderer::instance().context(), cache_->scene, 1, r, &id, &t, pos, nrm) != RTB_OK || id < 0)
        return res;
    res.hit = true;
    res.id = id;
    res.geometry = resolveHit(id);
    res.distance = t;
    res.position = Point(pos[0], pos[1], pos[2]);
    res.normal = Vector(nrm[0], nrm[1], nrm[2]);
    return res;
}

bool GeometrySet::intersectBatch(const float *rays, int64_t n, int32_t *hitId, float *hitT, float *position, float *normal)
{
    Ray probe(Point(0, 0, 0), Vector(0, 0, 1));
    rtb_scene *dev = uploadGeometry(*this);
    if (!dev) return false;
    rtb_ctx *ctx = CudaRenderer::instance().context();
    const int rc = rtb_intersect_rays(ctx, dev, n, rays, hitId, hitT, position, normal);
    rtb_scene_free(ctx, dev);
    return rc == RTB_OK;
}

// ---- PerformanceTest ------------------------------------------------------------------------------------
static Ptr<Material> solid(const Color &local, const Color &emission, float d, float r, float t)
{
    return Ptr<Material>(new SolidColorMaterial(local, emission, d, r, t));
}

Camera::Camera(const Point &eye, Vector front, const Vector &up)
{ // PerformanceTest/Camera.cpp:5-13
    this->eye = eye;
    this->front = front.norm();
    this->right = front.cross(up).norm();
    this->up = right.cross(front).norm();
}

Ray Camera::generateRay(float x, float y) const
{ // PerformanceTest/Camera.cpp:15-21
    const Vector r = right * ((x - 0.5f) * 1.274f);
    const Vector u = up * ((y - 0.5f) * 1.0f);
    Vector dir = front + r + u;
    dir.norm();
    return Ray(eye, dir);
}

// main.cpp:61-81: the tunnel (that program's own generator and k-d builder) and the plane closing its exit
Tunnel *PerformanceTest::buildScene(GeometrySet &scene, float pathRadius, float pathAngle, int archSeg, int pathSeg,
                                    Tunnel::Algorithm algorithm)
{
    scene.clear();
    TunnelGenerator g;
    g.performanceTestVariant = true;
    Ptr<Material> plain = solid(Color::Black(), Color::Black(), 1, 0, 0); // PerformanceTest has no materials
    g.create(50, 25, 25, pathRadius, pathAngle, archSeg, pathSeg, scene, plain, plain, algorithm);
    Tunnel *tunnel = static_cast<Tunnel *>(scene.last());
    const Vector normal(std::sin(pathAngle), 0, -std::cos(pathAngle)); // main.cpp:71-78
    Plane *exitPlane = new Plane(normal, pathRadius * std::sin(pathAngle));
    exitPlane->material = plain;
    scene.add(exitPlane);
    return tunnel;
}

bool PerformanceTest::build(float pathRadius, float pathAngle, int archSeg, int pathSeg, Tunnel::Algorithm algorithm)
{
    const double t0 = nowMs();
    tunnel = buildScene(scene, pathRadius, pathAngle, archSeg, pathSeg, algorithm);
    buildMs = nowMs() - t0;
    const double t1 = nowMs();
    tunnel->init();
    preprocessMs = nowMs() - t1;
    return true;
}

double PerformanceTest::run(const float *xy, int n, int maxDepth, int32_t *reached, int32_t *depth, int32_t *lastId,
                            float *lastPos, int64_t *totalRays)
{
    rtb_ctx *ctx = CudaRenderer::instance().context();
    if (!ctx) return -1;
    const Camera camera(Point(0, 25, 5), Vector(0, 0, -1), Vector(0, 1, 0)); // main.cpp:143-147
    std::vector<float> rays((size_t)n * 6);
    for (int i = 0; i < n; i++)
    {
        const Ray r = camera.generateRay(xy[2 * i], xy[2 * i + 1]);
        float *o = &rays[6 * (size_t)i];
        o[0] = r.origin.x; o[1] = r.origin.y; o[2] = r.origin.z;
        o[3] = r.direction.x; o[4] = r.direction.y; o[5] = r.direction.z;
    }
    FlatScene flat;
    scene.flatten(flat);
    flat.finish();
    rtb_scene *dev = nullptr;
    if (rtb_scene_upload(ctx, &flat.view, &dev) != RTB_OK) return -2;
    float ms = 0;
    const int rc = rtb_bounce_rays(ctx, dev, n, rays.data(), maxDepth, reached, depth, lastId, lastPos, totalRays, &ms);
    rtb_scene_free(ctx, dev);
    return rc == RTB_OK ? (double)ms : -3.0;
}

// ---- preset scene scripts (reference Scripts.cpp:22-278) ----------------------------------------
static void addCornellBox(GeometrySet &scene)
{ // the smallpt box of presets 2 and 3: six planes and the r=600 light sphere
    const struct { Vector n; float d; Color c; } walls[6] = {
        {Vector(1, 0, 0), 1, Color(0.75f, 0.25f, 0.25f)}, {Vector(1, 0, 0), 99, Color(0.25f, 0.25f, 0.75f)},
        {Vector(0, 1, 0), 0, Color(0.75f, 0.75f, 0.75f)}, {Vector(0, 1, 0), 81.6f, Color(0.75f, 0.75f, 0.75f)},
        {Vector(0, 0, 1), 0, Color(0.75f, 0.75f, 0.75f)}, {Vector(0, 0, 1), 170, Color(0, 0, 0)}};
    for (const auto &w : walls)
    {
        Plane *p = new Plane(w.n, w.d);
        p->material = solid(w.c, Color::Black(), 1, 0, 0);
        scene.add(p);
    }
    Sphere *light = new Sphere(Point(50, 681.6f - 0.27f, 81.6f), 600);
    light->material = solid(Color::Black(), Color(24, 24, 24), 1, 0, 0);
    scene.add(light);
}

bool Script::Build(GeometrySet &scene, std::unique_ptr<PerspectiveCamera> &camera, RenderSetting &setting,
                   int tunnelAlgorithm, int &prepareTime) const
{
    prepareTime = 0;
    if (preset == 1)
    {
        Plane *ground = new Plane(Vector(0, 1, 0), 0);
        ground->material = Ptr<Material>(new RadianceCheckerMaterial(1.2f, 0.025f));
        scene.add(ground);
        Sphere *s1 = new Sphere(Point(-10, 15, -30), 15), *s2 = new Sphere(Point(20, 10, -20), 10);
        s1->material = solid(Color::White(), Color::Black(), 1, 0, 0);
        s2->material = solid(Color::White(), Color::Black(), 1, 0, 0);
        scene.add(s1);
        scene.add(s2);
        camera.reset(new PerspectiveCamera(Point(0, 15, 30), Vector(0, 0, -1), Vector(0, 1, 0), 1.3333f, 65, 0));
        setting = RenderSetting::Default();
        return true;
    }
    if (preset == 2 || preset == 3)
    {
        addCornellBox(scene);
        if (preset == 2)
        {
            Sphere *mirror = new Sphere(Point(27, 16.5f, 47), 16.5f), *glass = new Sphere(Point(73, 16.5f, 78), 16.5f);
            mirror->material = solid(Color::White(), Color::Black(), 0, 1, 0);
            glass->material = Ptr<Material>(new GlassMaterial());
            scene.add(mirror);
            scene.add(glass);
        }
        else if (stlAsMeshDefault ? !scene.addStlMesh(stlPath.c_str(), Ptr<Material>(new GlassMaterial()), Matrix(1, 0, 0, 0, 1, 0, 0, 0, 1),
                                                      Vector(50, 0, 40))
                                  : !scene.addStlFile(stlPath.c_str(), Ptr<Material>(new GlassMaterial()), Matrix(1, 0, 0, 0, 1, 0, 0, 0, 1),
                                                      Vector(50, 0, 40)))
            return false;
        camera.reset(new PerspectiveCamera(Point(50, 52, 295), Vector(0, -0.045f, -1), Vector(0, 1, -0.045f), 1.3333f, 28, 140.0f));
        setting = RenderSetting::Default();
        return true;
    }
    // presets 4 (short wide tunnel) and 5 (long narrow tunnel)
    const bool wide = preset == 4;
    Sphere *ball = new Sphere(wide ? Point(74.12f, 15, -96.59f) : Point(5000, 15, -5000), 15);
    ball->material = Ptr<Material>(new PhongMaterial(Color(1, 0, 0), Color::White(), 16));
    scene.add(ball);
    Plane *ground = new Plane(Vector(0, 1, 0), -0.01f);
    ground->material = solid(Color(0.25, 0.25, 0.25), Color::Black(), 1, 0, 0);
    scene.add(ground);
    Plane *sky = new Plane(Vector(0, 1, 0), 1000);
    sky->material = solid(Color::White(), Color::Black(), 1, 0, 0);
    scene.add(sky);
    TunnelGenerator g;
    g.create(50, 25, 25, wide ? 100.0f : 5000.0f, wide ? PI * 0.416667f : PI * 0.5f, tunnelSegments, tunnelSegments, scene,
             Ptr<Material>(new CheckerMaterial(0.05f)), solid(Color::Black(), Color::Black(), 0.333f, 0.667f, 0),
             (Tunnel::Algorithm)tunnelAlgorithm);
    const double t1 = nowMs();
    static_cast<Tunnel *>(scene.last())->init();
    prepareTime = (int)(nowMs() - t1 + 0.5);
    camera.reset(new PerspectiveCamera(Point(0, 25, 20), Vector(0, 0, -1), Vector(0, 1, 0), 1.3333f, 65, 0.0f));
    setting = RenderSetting::Simple();
    return true;
}

void Script::Run(RenderProc render, int tunnelAlgorithm, LogCallback log, ProgressCallback progress, int &prepareTime,
                 int &execTime)
{
    GeometrySet scene;
    std::unique_ptr<PerspectiveCamera> camera;
    RenderSetting setting = RenderSetting::Simple();
    if (!Build(scene, camera, setting, tunnelAlgorithm, prepareTime))
    {
        if (log) log("Script: cannot build the scene (missing STL file?)\r\n");
        execTime = -1;
        return;
    }
    execTime = render(scene, *camera, setting, progress);
}

bool Script::stlAsMeshDefault = false;

static Script s1("checker ground and balls", Script::FLAG_MONTE_CARLO, 0, 1000, 1);
static Script s2("smallpt", Script::FLAG_MONTE_CARLO, 0, 1000, 2);
static Script s3("smallpt (stl)", Script::FLAG_MONTE_CARLO, 0, 1000, 3);
static Script s4("tunnel (short and wide)", Script::FLAG_TUNNEL, 150, 0, 4);
static Script s5("tunnel (long and narrow)", Script::FLAG_TUNNEL, 150, 0, 5);
Script *scripts[5] = {&s1, &s2, &s3, &s4, &s5};

} // namespace rt

// ---- C API for the Python harness ----------------------------------------------------------------
using namespace rt;

struct rtbh_scene
{
    GeometrySet scene;
    std::unique_ptr<PerspectiveCamera> camera;
    RenderSetting setting;
    FlatScene flat;
    rtb_camera cam;
    rtb_render_setting rs;
    int prepareMs = 0;
    double buildMs = 0, flattenMs = 0;
    Tunnel *tunnel = nullptr;
};

static inline void hmix(uint64_t &h, uint32_t v) { h = (h ^ v) * 0x100000001b3ull; }
static inline uint32_t fbits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }

extern "C" {

// Build preset `preset` (1..5, reference Scripts.cpp) with the host builders and flatten it.
rtbh_scene *rtbh_preset_create(int preset, int algorithm, int segments, const char *stl_path)
{
    if (preset < 1 || preset > 5 || algorithm < 0 || algorithm > 6) return nullptr;
    rtbh_scene *h = new rtbh_scene();
    Script script = *scripts[preset - 1];
    script.tunnelSegments = segments;
    if (stl_path) script.stlPath = stl_path;
    const double t0 = nowMs();
    if (!script.Build(h->scene, h->camera, h->setting, algorithm, h->prepareMs)) { delete h; return nullptr; }
    h->buildMs = nowMs() - t0;
    const double t1 = nowMs();
    h->scene.flatten(h->flat);
    h->flat.finish();
    h->flattenMs = nowMs() - t1;
    h->cam = h->camera->flatten();
    h->rs = h->setting.flatten();
    if (preset >= 4) h->tunnel = static_cast<Tunnel *>(h->scene.last());
    return h;
}
// The PerformanceTest scene (tunnel + exit plane, src/PerformanceTest/main.cpp:61-81) built and flattened; the
// handle serves the same queries as a preset's (stats, hashes, flat view) -- no camera / setting of its own.
rtbh_scene *rtbh_perf_scene_create(float radius, float angle, int arch_seg, int path_seg, int algorithm)
{
    if (algorithm < 0 || algorithm > 6 || arch_seg < 1 || path_seg < 1) return nullptr;
    rtbh_scene *h = new rtbh_scene();
    const double t0 = nowMs();
    h->tunnel = PerformanceTest::buildScene(h->scene, radius, angle, arch_seg, path_seg, (Tunnel::Algorithm)algorithm);
    const double t1 = nowMs();
    h->tunnel->init();
    h->prepareMs = (int)(nowMs() - t1);
    h->buildMs = nowMs() - t0;
    h->scene.flatten(h->flat);
    h->flat.finish();
    h->camera.reset(new PerspectiveCamera(Point(0, 25, 5), Vector(0, 0, -1), Vector(0, 1, 0), 1.274f, 53.13f, 0.0f));
    h->setting = RenderSetting::Simple();
    h->cam = h->camera->flatten();
    h->rs = h->setting.flatten();
    return h;
}
// tunnels generated from now on leave their grid to the device builder (Tunnel::gridOnDevice)
void rtbh_set_grid_on_device(int on) { Tunnel::gridOnDeviceDefault = on != 0; }
// ... bin their triangles with the exact overlap test (Tunnel::exactGridBinning)
void rtbh_set_exact_grid_binning(int on) { Tunnel::exactGridBinningDefault = on != 0; }
// ... leave their SAH k-d tree to the device builder (Tunnel::kdOnDevice)
void rtbh_set_kd_on_device(int on) { Tunnel::kdOnDeviceDefault = on != 0; }
// preset 3 built from now on loads its STL as one mesh (GeometrySet::addStlMesh) instead of loose triangles
void rtbh_set_stl_as_mesh(int on) { Script::stlAsMeshDefault = on != 0; }
void rtbh_free(rtbh_scene *h) { delete h; }
const rtb_flat_scene *rtbh_flat(const rtbh_scene *h) { return &h->flat.view; }
const rtb_camera *rtbh_camera(const rtbh_scene *h) { return &h->cam; }
const rtb_render_setting *rtbh_setting(const rtbh_scene *h) { return &h->rs; }
double rtbh_prepare_ms(const rtbh_scene *h) { return h->prepareMs; }
double rtbh_build_ms(const rtbh_scene *h) { return h->buildMs; }
int64_t rtbh_host_bytes(const rtbh_scene *h) { return (int64_t)h->flat.hostBytes(); }

// stats in the order of oracle_abi.h's ORACLE_STAT_* (n_top, n_tris, grid xyz, cells, entries, max, kd nodes, leaves, refs, depth)
void rtbh_stats(const rtbh_scene *h, int64_t *out)
{
    memset(out, 0, 16 * sizeof(int64_t));
    out[0] = h->flat.view.n_top;
    out[1] = h->flat.view.n_tris;
    if (h->tunnel)
    {
        const Tunnel::BuildStats &s = h->tunnel->stats;
        out[2] = s.gridX; out[3] = s.gridY; out[4] = s.gridZ;
        out[5] = s.cellsNonEmpty; out[6] = s.cellEntries; out[7] = s.cellMax;
        out[8] = s.kdNodes; out[9] = s.kdLeaves; out[10] = s.kdLeafRefs; out[11] = s.kdMaxDepth;
    }
}

// canonical digest of the tunnel triangle stream (a, b, c, normal, ground flag)
uint64_t rtbh_tri_hash(const rtbh_scene *h)
{
    const rtb_flat_scene &f = h->flat.view;
    if (f.n_tris == 0) return 0;
    uint64_t x = 0xcbf29ce484222325ull;
    const int groundMat = f.tri_material[f.n_tris - 1];
    for (int k = 0; k < f.n_tris; k++)
    {
        for (int q = 0; q < 12; q++) hmix(x, fbits(f.tri[12 * (size_t)k + q]));
        hmix(x, f.tri_material[k] == groundMat ? 1u : 0u);
    }
    return x;
}

// canonical digest of the flattened accelerator, computed from the FLAT buffers: walks the sparse
// cell directory / the pre-order node array exactly as the kernels read them
uint64_t rtbh_struct_hash(const rtbh_scene *h)
{
    const rtb_flat_scene &f = h->flat.view;
    uint64_t x = 0xcbf29ce484222325ull;
    if (f.n_tris == 0) return 0;
    if (f.accel == RTB_ACCEL_REGULAR_GRID || f.accel == RTB_ACCEL_FLAT_GRID)
    {
        hmix(x, 0x47524944u);
        for (int a = 0; a < 3; a++) hmix(x, (uint32_t)f.grid_dims[a]);
        for (int a = 0; a < 3; a++) hmix(x, fbits(f.grid_origin[a]));
        for (int a = 0; a < 3; a++) hmix(x, fbits(f.grid_cell[a]));
        for (int64_t w = 0; w < f.n_cellwords; w++)
        {
            uint32_t bits = f.grid_words[w].bits, r = f.grid_words[w].rank;
            while (bits)
            {
                const int b = __builtin_ctz(bits);
                bits &= bits - 1;
                const uint32_t first = f.grid_cell_start[r], last = f.grid_cell_start[r + 1];
                hmix(x, (uint32_t)(w * 32 + b));
                hmix(x, last - first);
                for (uint32_t e = first; e < last; e++) hmix(x, f.grid_cell_tris[e]);
                r++;
            }
        }
        return x;
    }
    if (f.accel == RTB_ACCEL_CONVEX || f.accel == RTB_ACCEL_CONVEX_SIMPLE)
    { // convex accelerator tables, same convention as oracle/rt_oracle.cpp and oracle/ref/ref_pt_driver.cpp
        if (!f.cx_frames) return 0;
        hmix(x, 0x43565800u);
        hmix(x, (uint32_t)f.n_cx_path); hmix(x, (uint32_t)f.n_cx_edges);
        hmix(x, fbits(f.cx_width)); hmix(x, fbits(f.cx_height));
        for (int i = 0; i < f.n_cx_path * 8; i++) hmix(x, fbits(f.cx_frames[i]));
        for (int i = 0; i < f.n_cx_edges * 3; i++) hmix(x, fbits(f.cx_edges[i]));
        const int cells = f.cx_table_size * f.cx_table_size;
        for (int i = 0; i < cells; i++) hmix(x, f.cx_cell_status[i]);
        for (int i = 0; i < cells * 2; i++) hmix(x, (uint32_t)(uint16_t)f.cx_cell_range[i]);
        if (f.accel == RTB_ACCEL_CONVEX)
            for (int64_t i = 0; i < (int64_t)100 * 360 * 2 * f.n_cx_edges; i++) hmix(x, f.cx_order[i]);
        return x;
    }
    if (f.accel == RTB_ACCEL_KD_MEDIAN || f.accel == RTB_ACCEL_KD_SAH)
    {
        hmix(x, 0x4b445452u);
        for (int a = 0; a < 3; a++) hmix(x, fbits(f.kd_min[a]));
        for (int a = 0; a < 3; a++) hmix(x, fbits(f.kd_max[a]));
        for (int i = 0; i < f.n_kd_nodes; i++) // array order IS pre-order
        {
            const rtb_kdnode &n = f.kd_nodes[i];
            if ((n.b & 3u) == 3u)
            {
                hmix(x, 3);
                hmix(x, n.b >> 2);
                for (uint32_t e = 0; e < (n.b >> 2); e++) hmix(x, f.kd_leaf_tris[n.a + e]);
            }
            else { hmix(x, n.b & 3u); hmix(x, n.a); }
        }
        return x;
    }
    return 0;
}

// The drop-in path end to end: Script::Run(CudaRenderer::Render, ...) exactly as the reference's
// RenderThread calls it (MainWindow.cpp:369).  rgb_out (may be NULL): w*h*3 floats, reference order.
int rtbh_script_run(int preset, int algorithm, int segments, int width, int height, int samples, uint64_t seed,
                    int device, const char *stl_path, float *rgb_out, int *prepare_ms, int *exec_ms, rtb_stats *stats)
{
    if (preset < 1 || preset > 5) return -1;
    CudaRenderer &r = CudaRenderer::instance();
    r.configure(width, height, samples, device, seed);
    Script script = *scripts[preset - 1];
    script.tunnelSegments = segments;
    script.samples = samples;
    if (stl_path) script.stlPath = stl_path;
    int prep = 0, exec = 0;
    script.Run(CudaRenderer::Render, algorithm, nullptr, nullptr, prep, exec);
    if (prepare_ms) *prepare_ms = prep;
    if (exec_ms) *exec_ms = exec;
    if (exec < 0) return exec;
    if (rgb_out) memcpy(rgb_out, r.image().data(), r.image().size() * sizeof(float));
    if (stats) *stats = r.stats();
    return 0;
}

// The same path with everything a caller of the reference can observe: `n_devices` GPUs behind the one RenderProc,
// the ProgressCallback (calls counted, monotone, last value) and the LogCallback (text collected into log_out).
static int g_progressCalls = 0, g_progressLast = 0, g_progressTotal = 0, g_progressMonotone = 1;
static std::string g_logText;
static void countingProgress(int cur, int total)
{
    if (cur < g_progressLast) g_progressMonotone = 0;
    g_progressCalls++; g_progressLast = cur; g_progressTotal = total;
}
static void collectingLog(const char *str) { g_logText += str; }

int rtbh_script_run_ex(int preset, int algorithm, int segments, int width, int height, int samples, uint64_t seed, int device,
                       int n_devices, const char *stl_path, float *rgb_out, int *exec_ms, rtb_stats *stats, int progress_out[4],
                       char *log_out, int log_cap)
{
    if (preset < 1 || preset > 5) return -1;
    CudaRenderer &r = CudaRenderer::instance();
    r.configure(width, height, samples, device, seed);
    r.setDevices(n_devices);
    r.setLog(collectingLog);
    g_progressCalls = 0; g_progressLast = 0; g_progressTotal = 0; g_progressMonotone = 1;
    g_logText.clear();
    Script script = *scripts[preset - 1];
    script.tunnelSegments = segments;
    script.samples = samples;
    if (stl_path) script.stlPath = stl_path;
    int prep = 0, exec = 0;
    script.Run(CudaRenderer::Render, algorithm, collectingLog, countingProgress, prep, exec);
    r.setDevices(1);
    r.setLog(nullptr);
    if (exec_ms) *exec_ms = exec;
    if (progress_out) { progress_out[0] = g_progressCalls; progress_out[1] = g_progressLast; progress_out[2] = g_progressTotal; progress_out[3] = g_progressMonotone; }
    if (log_out && log_cap > 0) { strncpy(log_out, g_logText.c_str(), (size_t)log_cap - 1); log_out[log_cap - 1] = 0; }
    if (exec < 0) return exec;
    if (rgb_out) memcpy(rgb_out, r.image().data(), r.image().size() * sizeof(float));
    if (stats) *stats = r.stats();
    return 0;
}

// Same drop-in path with the 8-bit output stage; optionally writes a BMP (Save-As).
int rtbh_script_run8(int preset, int algorithm, int segments, int width, int height, int samples, uint64_t seed, int device,
                     const char *stl_path, unsigned char *rgb8_out, const char *bmp_path, int *exec_ms, rtb_stats *stats)
{
    if (preset < 1 || preset > 5) return -1;
    CudaRenderer &r = CudaRenderer::instance();
    r.configure(width, height, samples, device, seed);
    r.setOutput8bit(true);
    Script script = *scripts[preset - 1];
    script.tunnelSegments = segments;
    script.samples = samples;
    if (stl_path) script.stlPath = stl_path;
    int prep = 0, exec = 0;
    script.Run(CudaRenderer::Render, algorithm, nullptr, nullptr, prep, exec);
    r.setOutput8bit(false);
    if (exec_ms) *exec_ms = exec;
    if (exec < 0) return exec;
    if (rgb8_out) memcpy(rgb8_out, r.pixels().data(), r.pixels().size());
    if (stats) *stats = r.stats();
    if (bmp_path && !r.saveBitmap(bmp_path)) return -5;
    return 0;
}

// PerformanceTest console benchmark: `PerformanceTest radius angle archSeg pathSeg N algorithm` (main.cpp:83-125)
int rtbh_perf_test(float radius, float angle, int arch_seg, int path_seg, int algorithm, int n, const float *xy, int max_depth,
                   int32_t *reached, int32_t *depth, int32_t *last_id, float *last_pos, int64_t *total_rays,
                   double *build_ms, double *preprocess_ms, double *trace_ms)
{
    if (algorithm < 0 || algorithm > 6) return -1;
    PerformanceTest pt;
    pt.build(radius, angle, arch_seg, path_seg, (Tunnel::Algorithm)algorithm);
    const double ms = pt.run(xy, n, max_depth, reached, depth, last_id, last_pos, total_rays);
    if (build_ms) *build_ms = pt.buildMs;
    if (preprocess_ms) *preprocess_ms = pt.preprocessMs;
    if (trace_ms) *trace_ms = ms;
    return ms < 0 ? (int)ms : 0;
}

const char *rtbh_last_error() { return CudaRenderer::instance().lastError().c_str(); }

// Geometry::intersect / GeometrySet::intersectBatch through the host API (GPU-served)
int rtbh_intersect_batch(rtbh_scene *h, int64_t n, const float *rays, int32_t *hit_id, float *hit_t, float *position,
                         float *normal)
{
    return h->scene.intersectBatch(rays, n, hit_id, hit_t, position, normal) ? 0 : -1;
}
int rtbh_intersect_one(rtbh_scene *h, const float *ray6, int32_t *hit_id, float *hit_t, float *position, float *normal)
{
    Ray r(Point(ray6[0], ray6[1], ray6[2]), Vector(ray6[3], ray6[4], ray6[5]));
    IntersectResult res = h->scene.intersect(r);
    *hit_id = res.hit ? res.id : -1;
    *hit_t = res.hit ? res.distance : -1.0f;
    if (position) { position[0] = res.position.x; position[1] = res.position.y; position[2] = res.position.z; }
    if (normal) { normal[0] = res.normal.x; normal[1] = res.normal.y; normal[2] = res.normal.z; }
    return 0;
}

} // extern "C"
