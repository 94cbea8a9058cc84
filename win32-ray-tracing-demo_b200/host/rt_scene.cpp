// rt_scene.cpp -- materials, geometries, camera: parameter carriers and their flatten() to the
// SoA buffers of include/rtb.h.  No intersection or shading arithmetic lives on the host.
#include "rt.h"

#include <cstdio>
#include <cstring>
#include <mutex>

namespace rt {

// ---- materials --------------------------------------------------------------------------------
rtb_material Material::base(int kind) const
{
    rtb_material m;
    memset(&m, 0, sizeof(m));
    m.kind = kind;
    m.diffusiveness = diffusiveness;
    m.reflectiveness = reflectiveness;
    m.refractiveness = refractiveness;
    m.refractive_index = refractive_index;
    return m;
}

rtb_material SolidColorMaterial::flatten() const
{
    rtb_material m = base(RTB_MAT_SOLID);
    m.a[0] = localColor.r; m.a[1] = localColor.g; m.a[2] = localColor.b;
    m.b[0] = emissionColor.r; m.b[1] = emissionColor.g; m.b[2] = emissionColor.b;
    return m;
}

static int flatDir(int d) { return d == 0 ? RTB_DIR_XOZ : (d == 1 ? RTB_DIR_XOY : RTB_DIR_YOZ); }

rtb_material CheckerMaterial::flatten() const
{
    rtb_material m = base(RTB_MAT_CHECKER);
    m.scale = scale;
    m.dir = flatDir((int)dir);
    return m;
}

rtb_material RadianceCheckerMaterial::flatten() const
{
    rtb_material m = base(RTB_MAT_RADIANCE_CHECKER);
    m.scale = scale;
    m.p = radiance;
    m.dir = flatDir((int)dir);
    return m;
}

rtb_material PhongMaterial::flatten() const
{
    rtb_material m = base(RTB_MAT_PHONG);
    m.a[0] = diffuse.r; m.a[1] = diffuse.g; m.a[2] = diffuse.b;
    m.b[0] = specular.r; m.b[1] = specular.g; m.b[2] = specular.b;
    m.p = shininess;
    return m;
}

// ---- FlatScene --------------------------------------------------------------------------------
FlatScene::FlatScene() { memset(&view, 0, sizeof(view)); }

int FlatScene::materialIndex(const Material *m)
{
    for (size_t i = 0; i < materialKeys.size(); i++)
        if (materialKeys[i] == m) return (int)i;
    materialKeys.push_back(m);
    materials.push_back(m->flatten());
    return (int)materials.size() - 1;
}

void FlatScene::finish()
{
    view.n_prims = (int32_t)prims.size(); view.prims = prims.data();
    view.n_materials = (int32_t)materials.size(); view.materials = materials.data();
    view.n_top = nTop;
    view.n_loose = (int32_t)(looseTri.size() / 12); view.loose_tri = looseTri.empty() ? nullptr : looseTri.data();
    view.n_tris = (int32_t)(tri.size() / 12); view.tri = tri.empty() ? nullptr : tri.data();
    view.tri_material = triMaterial.empty() ? nullptr : triMaterial.data();
    view.n_cellwords = (int64_t)gridWords.size(); view.grid_words = gridWords.empty() ? nullptr : gridWords.data();
    view.n_cells_used = gridCellStart.empty() ? 0 : (int64_t)gridCellStart.size() - 1;
    view.grid_cell_start = gridCellStart.empty() ? nullptr : gridCellStart.data();
    view.n_cell_refs = (int64_t)gridCellTris.size(); view.grid_cell_tris = gridCellTris.empty() ? nullptr : gridCellTris.data();
    view.n_kd_nodes = (int32_t)kdNodes.size(); view.kd_nodes = kdNodes.empty() ? nullptr : kdNodes.data();
    view.n_kd_refs = (int64_t)kdLeafTris.size(); view.kd_leaf_tris = kdLeafTris.empty() ? nullptr : kdLeafTris.data();
    view.n_cx_path = (int32_t)(cxFrames.size() / 8); view.cx_frames = cxFrames.empty() ? nullptr : cxFrames.data();
    view.n_cx_edges = (int32_t)(cxEdges.size() / 3); view.cx_edges = cxEdges.empty() ? nullptr : cxEdges.data();
    view.cx_cell_status = cxCellStatus.empty() ? nullptr : cxCellStatus.data();
    view.cx_cell_range = cxCellRange.empty() ? nullptr : cxCellRange.data();
    view.cx_order = cxOrder.empty() ? nullptr : cxOrder.data();
}

size_t FlatScene::hostBytes() const
{
    return prims.size() * sizeof(rtb_prim) + materials.size() * sizeof(rtb_material) + (looseTri.size() + tri.size()) * 4 +
           triMaterial.size() * 4 + gridWords.size() * sizeof(rtb_cellword) + (gridCellStart.size() + gridCellTris.size()) * 4 +
           kdNodes.size() * sizeof(rtb_kdnode) + kdLeafTris.size() * 4 + (cxFrames.size() + cxEdges.size()) * 4 +
           cxCellStatus.size() + cxCellRange.size() * 2 + cxOrder.size() * 2;
}

// ---- geometries -------------------------------------------------------------------------------
static void pushTriangle(std::vector<float> &dst, const Point &a, const Point &b, const Point &c, const Vector &n)
{
    const float v[12] = {a.x, a.y, a.z, b.x, b.y, b.z, c.x, c.y, c.z, n.x, n.y, n.z};
    dst.insert(dst.end(), v, v + 12);
}

void Plane::flatten(FlatScene &out) const
{
    rtb_prim p;
    memset(&p, 0, sizeof(p));
    p.type = RTB_PRIM_PLANE;
    p.material = out.materialIndex(material.get());
    p.base_id = out.nTop++;
    p.v[0] = normal.x; p.v[1] = normal.y; p.v[2] = normal.z;
    p.v[3] = position.x; p.v[4] = position.y; p.v[5] = position.z;
    p.v[6] = dist;
    out.prims.push_back(p);
}

void Sphere::flatten(FlatScene &out) const
{
    rtb_prim p;
    memset(&p, 0, sizeof(p));
    p.type = RTB_PRIM_SPHERE;
    p.material = out.materialIndex(material.get());
    p.base_id = out.nTop++;
    p.v[0] = center.x; p.v[1] = center.y; p.v[2] = center.z;
    p.v[3] = radius;
    out.prims.push_back(p);
}

void Triangle::getBoundingBox(Point &mn, Point &mx) const
{
    mn = Point(std::fmin(std::fmin(a.x, b.x), c.x), std::fmin(std::fmin(a.y, b.y), c.y), std::fmin(std::fmin(a.z, b.z), c.z));
    mx = Point(std::fmax(std::fmax(a.x, b.x), c.x), std::fmax(std::fmax(a.y, b.y), c.y), std::fmax(std::fmax(a.z, b.z), c.z));
}

void Triangle::flatten(FlatScene &out) const
{
    // consecutive loose triangles sharing a material extend the previous run record
    const int mat = out.materialIndex(material.get());
    const int index = (int)(out.looseTri.size() / 12);
    pushTriangle(out.looseTri, a, b, c, normal);
    const int id = out.nTop++;
    if (!out.prims.empty())
    {
        rtb_prim &last = out.prims.back();
        if (last.type == RTB_PRIM_TRIANGLES && last.material == mat && last.first + last.count == index &&
            last.base_id + last.count == id)
        {
            last.count++;
            return;
        }
    }
    rtb_prim p;
    memset(&p, 0, sizeof(p));
    p.type = RTB_PRIM_TRIANGLES;
    p.material = mat;
    p.base_id = id;
    p.first = index;
    p.count = 1;
    out.prims.push_back(p);
}

void TriangleMesh::add(const Point &a, const Point &b, const Point &c, const Vector &normal)
{
    pushTriangle(tris, a, b, c, normal);
    invalidate();
}

void TriangleMesh::flatten(FlatScene &out) const
{
    if (tris.empty()) return;
    rtb_prim p;
    memset(&p, 0, sizeof(p));
    p.type = RTB_PRIM_MESH;
    p.material = out.materialIndex(material.get());
    p.base_id = out.nTop;
    p.first = (int)(out.looseTri.size() / 12);
    p.count = (int)count();
    out.looseTri.insert(out.looseTri.end(), tris.begin(), tris.end());
    out.nTop += p.count;
    out.prims.push_back(p);
}

GeometrySet::~GeometrySet() { clear(); }

void GeometrySet::clear()
{
    for (Geometry *g : geometries) delete g;
    geometries.clear();
    variableIds_ = false;
    invalidate();
}

bool GeometrySet::addStlFile(const char *filename, Ptr<Material> material)
{
    return addStlFile(filename, material, Matrix(1, 0, 0, 0, 1, 0, 0, 0, 1), Vector(0, 0, 0));
}

// binary STL: 80-byte header, u32 count, then per facet 12 floats + u16 (reference GeometrySet.cpp:33-86); `facet` receives
// the transformed vertices and normal of every facet
template <class Facet>
static bool readStl(const char *filename, const Matrix &matrix, const Vector &offset, Facet facet)
{
    FILE *fp = fopen(filename, "rb");
    if (!fp) return false;
    unsigned char header[84];
    if (fread(header, 1, 84, fp) != 84) { fclose(fp); return false; }
    uint32_t count;
    memcpy(&count, header + 80, 4);
    std::vector<unsigned char> body((size_t)count * 50);
    const bool ok = fread(body.data(), 1, body.size(), fp) == body.size();
    fclose(fp);
    if (!ok) return false;
    for (uint32_t i = 0; i < count; i++)
    {
        float f[12];
        memcpy(f, body.data() + (size_t)i * 50, 48);
        const Point p1 = matrix * Point(f[3], f[4], f[5]) + offset;
        const Point p2 = matrix * Point(f[6], f[7], f[8]) + offset;
        const Point p3 = matrix * Point(f[9], f[10], f[11]) + offset;
        const Vector n = matrix * Vector(f[0], f[1], f[2]).norm();
        facet(p1, p2, p3, n);
    }
    return true;
}

bool GeometrySet::addStlFile(const char *filename, Ptr<Material> material, const Matrix &matrix, const Vector &offset)
{
    const bool ok = readStl(filename, matrix, offset, [&](const Point &p1, const Point &p2, const Point &p3, const Vector &n) {
        Triangle *t = new Triangle(p1, p2, p3, n);
        t->material = material;
        geometries.push_back(t);
    });
    if (ok) invalidate();
    return ok;
}

bool GeometrySet::addStlMesh(const char *filename, Ptr<Material> material)
{
    return addStlMesh(filename, material, Matrix(1, 0, 0, 0, 1, 0, 0, 0, 1), Vector(0, 0, 0));
}

bool GeometrySet::addStlMesh(const char *filename, Ptr<Material> material, const Matrix &matrix, const Vector &offset)
{
    TriangleMesh *mesh = new TriangleMesh();
    mesh->material = material;
    if (!readStl(filename, matrix, offset, [&](const Point &p1, const Point &p2, const Point &p3, const Vector &n) { mesh->add(p1, p2, p3, n); }))
    {
        delete mesh;
        return false;
    }
    add(mesh);
    return true;
}

void GeometrySet::flatten(FlatScene &out) const
{
    for (const Geometry *g : geometries) g->flatten(out);
}

// ---- camera -----------------------------------------------------------------------------------
PerspectiveCamera::PerspectiveCamera(const Point &eye, Vector front, const Vector &up, float ratio, float fov, float forward)
{ // reference Camera.cpp:4-18; `front` is normalised before right/up are derived from it
    this->eye = eye;
    this->front = front.norm();
    this->ratio = ratio;
    this->fov = fov;
    this->forward = forward;
    this->right = front.cross(up).norm();
    this->up = right.cross(front).norm();
    this->xcenter = ratio * 0.5f;
    this->fovScale = std::tan(fov * (PI * 0.5f / 180)) * 2;
}

Ray PerspectiveCamera::generateRay(float x, float y) const
{
    const Vector r = right * ((x - xcenter) * fovScale);
    const Vector u = up * ((y - 0.5f) * fovScale);
    Vector dir = (front + r + u);
    dir.norm();
    return Ray(eye + dir * forward, dir);
}

rtb_camera PerspectiveCamera::flatten() const
{
    rtb_camera c;
    memset(&c, 0, sizeof(c));
    c.eye[0] = eye.x; c.eye[1] = eye.y; c.eye[2] = eye.z;
    c.front[0] = front.x; c.front[1] = front.y; c.front[2] = front.z;
    c.up[0] = up.x; c.up[1] = up.y; c.up[2] = up.z;
    c.right[0] = right.x; c.right[1] = right.y; c.right[2] = right.z;
    c.xcenter = xcenter;
    c.fov_scale = fovScale;
    c.forward = forward;
    return c;
}

} // namespace rt
