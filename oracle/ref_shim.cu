// TEST INFRASTRUCTURE ONLY -- never linked into, loaded by, or shipped with the product.
//
// oracle/_ref/libptref.so: the reference's OWN __host__ __device__ functions, compiled
// for the host by nvcc from the sources where they lie under the reference checkout (nothing is
// copied into this repo).  This file only adds extern "C" batch wrappers so that Python
// (ctypes) can call them.  It is used for exactly two things:
//   1. oracle/gen_golden.py  -> writes tests/golden/*.json (the committed golden vectors)
//   2. tests/test_oracle_vs_ref.py (runs only where oracle/_ref exists) -> pins the C
//      restatement oracle/pt_oracle.c bit-for-bit against the reference's functions.
//
// Functions wrapped (reference file:line):
//   hash                                  src/intersections.h:26-34
//   multiplyMV                            src/intersections.h:53-59
//   getPointOnRay                         src/intersections.h:46-48
//   sphereIntersectionTest                src/intersections.h:81-117
//   boxIntersectionTest (stub, -1)        src/intersections.h:74-77
//   getRadiuses                           src/intersections.h:120-129
//   calculateRandomDirectionInHemisphere  src/interactions.h:62-87
//   calculateBSDF (stub, 1)               src/interactions.h:99-104
//   getRandomPointOnCube                  src/intersections.h:133-175 (host evaluation order of the reference build)
//   getRandomPointOnSphere (stub, 0)      src/intersections.h:179-182
//   calculateTransmission / getRandomDirectionInSphere (stubs, 0)   src/interactions.h:31-33,93-95
//
// intersections.h must come before any header that says `using namespace std`
// (SURVEY.md D9: ::hash vs std::hash).
#include "intersections.h"
#include "interactions.h"
#include <cstddef>
#include <cstring>

static_assert(sizeof(staticGeom) == 172, "staticGeom ABI");
static_assert(sizeof(material) == 64, "material ABI");
static_assert(sizeof(cameraData) == 52, "cameraData ABI");
static_assert(sizeof(ray) == 24, "ray ABI");

extern "C" {

unsigned int ref_hash(unsigned int a) { return ::hash(a); }

void ref_multiplyMV(const float* m16, const float* v4, float* out3) {
  cudaMat4 m;
  std::memcpy(&m, m16, 64);
  glm::vec3 r = multiplyMV(m, glm::vec4(v4[0], v4[1], v4[2], v4[3]));
  out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
}

void ref_getPointOnRay(const float* o3, const float* d3, float t, float* out3) {
  ray r; r.origin = glm::vec3(o3[0], o3[1], o3[2]); r.direction = glm::vec3(d3[0], d3[1], d3[2]);
  glm::vec3 p = getPointOnRay(r, t);
  out3[0] = p.x; out3[1] = p.y; out3[2] = p.z;
}

// nrays rays against ONE geom (172-byte staticGeom image). which: 0 sphere test, 1 box test.
void ref_intersect_batch(const void* geom172, int which, int nrays, const float* o, const float* d,
                         float* t, float* p, float* n) {
  staticGeom g;
  std::memcpy(&g, geom172, sizeof(g));
  for (int i = 0; i < nrays; i++) {
    ray r;
    r.origin = glm::vec3(o[3 * i], o[3 * i + 1], o[3 * i + 2]);
    r.direction = glm::vec3(d[3 * i], d[3 * i + 1], d[3 * i + 2]);
    glm::vec3 pp(0, 0, 0), nn(0, 0, 0);
    float tt = which == 0 ? sphereIntersectionTest(g, r, pp, nn) : boxIntersectionTest(g, r, pp, nn);
    t[i] = tt;
    p[3 * i] = pp.x; p[3 * i + 1] = pp.y; p[3 * i + 2] = pp.z;
    n[3 * i] = nn.x; n[3 * i + 1] = nn.y; n[3 * i + 2] = nn.z;
  }
}

void ref_getRadiuses(const void* geom172, float* out3) {
  staticGeom g;
  std::memcpy(&g, geom172, sizeof(g));
  glm::vec3 r = getRadiuses(g);
  out3[0] = r.x; out3[1] = r.y; out3[2] = r.z;
}

void ref_hemisphere_batch(int n, const float* normal, const float* xi1, const float* xi2, float* out) {
  for (int i = 0; i < n; i++) {
    glm::vec3 r = calculateRandomDirectionInHemisphere(
        glm::vec3(normal[3 * i], normal[3 * i + 1], normal[3 * i + 2]), xi1[i], xi2[i]);
    out[3 * i] = r.x; out[3 * i + 1] = r.y; out[3 * i + 2] = r.z;
  }
}

int ref_calculateBSDF_stub(void) {
  ray r; r.origin = glm::vec3(0); r.direction = glm::vec3(0, 0, -1);
  AbsorptionAndScatteringProperties a; a.absorptionCoefficient = glm::vec3(0); a.reducedScatteringCoefficient = 0;
  glm::vec3 c(0), u(0);
  material m; std::memset(&m, 0, sizeof(m));
  return calculateBSDF(r, glm::vec3(0), glm::vec3(0, 1, 0), glm::vec3(0), a, c, u, m);
}

// n seeds against ONE cube: the reference's own sampler (thrust minstd seeded with hash((uint)seed))
void ref_getRandomPointOnCube_batch(const void* geom172, int n, const float* seed, float* out) {
  staticGeom g;
  std::memcpy(&g, geom172, sizeof(g));
  for (int i = 0; i < n; i++) {
    glm::vec3 p = getRandomPointOnCube(g, seed[i]);
    out[3 * i] = p.x; out[3 * i + 1] = p.y; out[3 * i + 2] = p.z;
  }
}

// the small helpers: epsilonCheck :37-43, getInverseDirectionOfRay :62-64, getSignOfRay :67-70
int ref_epsilonCheck(float a, float b) { return epsilonCheck(a, b) ? 1 : 0; }
void ref_ray_helpers(const float* d3, float* inv3, float* sign3) {
  ray r; r.origin = glm::vec3(0); r.direction = glm::vec3(d3[0], d3[1], d3[2]);
  glm::vec3 a = getInverseDirectionOfRay(r), b = getSignOfRay(r);
  inv3[0] = a.x; inv3[1] = a.y; inv3[2] = a.z; sign3[0] = b.x; sign3[1] = b.y; sign3[2] = b.z;
}

// the stubs this repo specifies itself: what the reference returns today (all zeros)
void ref_sampling_stubs(float* out9) {
  staticGeom g; std::memset(&g, 0, sizeof(g));
  glm::vec3 a = getRandomPointOnSphere(g, 1.0f), b = getRandomDirectionInSphere(0.3f, 0.7f),
            c = calculateTransmission(glm::vec3(1, 2, 3), 1.0f);
  out9[0] = a.x; out9[1] = a.y; out9[2] = a.z; out9[3] = b.x; out9[4] = b.y; out9[5] = b.z;
  out9[6] = c.x; out9[7] = c.y; out9[8] = c.z;
}

// sizeof / offsetof table (SURVEY.md appendix B)
int ref_layout(int* out, int cap) {
  int v[] = {
      (int)sizeof(ray), (int)sizeof(geom), (int)sizeof(staticGeom), (int)sizeof(cameraData),
      (int)sizeof(camera), (int)sizeof(material), (int)sizeof(cudaMat4),
      (int)offsetof(staticGeom, type), (int)offsetof(staticGeom, materialid),
      (int)offsetof(staticGeom, translation), (int)offsetof(staticGeom, rotation),
      (int)offsetof(staticGeom, scale), (int)offsetof(staticGeom, transform),
      (int)offsetof(staticGeom, inverseTransform),
      (int)offsetof(cameraData, resolution), (int)offsetof(cameraData, position),
      (int)offsetof(cameraData, view), (int)offsetof(cameraData, up), (int)offsetof(cameraData, fov),
      (int)offsetof(material, color), (int)offsetof(material, specularExponent),
      (int)offsetof(material, specularColor), (int)offsetof(material, hasReflective),
      (int)offsetof(material, hasRefractive), (int)offsetof(material, indexOfRefraction),
      (int)offsetof(material, hasScatter), (int)offsetof(material, absorptionCoefficient),
      (int)offsetof(material, reducedScatterCoefficient), (int)offsetof(material, emittance),
      (int)offsetof(geom, type), (int)offsetof(geom, materialid), (int)offsetof(geom, frames),
      (int)offsetof(geom, translations), (int)offsetof(geom, rotations), (int)offsetof(geom, scales),
      (int)offsetof(geom, transforms), (int)offsetof(geom, inverseTransforms),
      (int)offsetof(camera, resolution), (int)offsetof(camera, positions), (int)offsetof(camera, views),
      (int)offsetof(camera, ups), (int)offsetof(camera, frames), (int)offsetof(camera, fov),
      (int)offsetof(camera, iterations), (int)offsetof(camera, image), (int)offsetof(camera, rayList),
      (int)offsetof(camera, imageName),
  };
  int n = (int)(sizeof(v) / sizeof(v[0]));
  for (int i = 0; i < n && i < cap; i++) out[i] = v[i];
  return n;
}

}  // extern "C"
