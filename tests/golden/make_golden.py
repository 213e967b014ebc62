"""Regenerates the golden fixtures in this directory FROM THE REFERENCE (run in the build container only:
needs /root/reference and the binaries built by `make -C oracle/ref`).

  kat.json            known-answer values printed by a ~60-line host program compiled against the reference's
                      own headers (hash32, PCG32, normalizedUint, sobol::sample, cosineHemisphere, Fresnel terms,
                      computeDiffuseFresnel, the tent filter CDF, TangentFrame)
  kat_bsdfs.json      eval / pdf / sample of the reference's own BSDF classes (nine parameterisations, 40 direction pairs and 40
                      draws each through its SobolPathSampler), from a host program linked against the reference's objects
  kat_lights.json     sampleDirect / intersect / directPdf / evalDirect of its Quad, TriangleMesh and InfiniteSphere (+ BitmapTexture
                      importance map) classes
  kat_instances.json  Instance transforms: fromMatrix / quaternion composition / pos + rot*p through its Mat4f and QuaternionF classes
  kat_curves.json     HairBcsdf eval / pdf / sample and Curves::intersect (400 rays at 6 strands) of its classes
  <scene>/            scene JSON + .wo3 written by tungsten_b200.synth, plus
  <scene>/ref_pathseed.pfm   framebuffer of oracle/_ref/tungsten_pathseed (per-path reseed contract)
  <scene>/ref_stock.pfm      framebuffer of the UNMODIFIED reference binary
  hair_sky/                  curves + hair BCSDF lit by the shipped hair scene's own emitters (infinite_sphere_cap + skydome);
                             scene_sky_top.pfm = the image Skydome::prepareForRender computed, dumped through the reference's
                             classes, down to the horizon (the 2:1 image is zero below it; tests pad it back: "scene_sky.pfm")
  cornell_adaptive/          the same with renderer.adaptive_sampling = true, 48 spp in three 16-spp steps
  materialtest/, hair_shipped/   shrunk copies of two scenes the reference ships + its renders of them (make_shipped_scenes)
  sobol_reference.json       checksum and sampled entries of the reference's Sobol direction matrices

The fixtures are small (64x64) so that the CPU test-suite stays fast; they travel to the GPU box with the
repository, /root/reference does not.
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"

KAT_CPP = r'''
#include <cstdio>
#include <cmath>
#include "math/MathUtil.hpp"
#include "math/BitManip.hpp"
#include "math/TangentFrame.hpp"
#include "sampling/UniformSampler.hpp"
#include "sampling/SampleWarp.hpp"
#include "bsdfs/Fresnel.hpp"
#include "bsdfs/Microfacet.hpp"
#include <sobol/sobol.h>
using namespace Tungsten;
static void pf(const char *k, float v, bool last = false) { union { float f; unsigned u; } c; c.f = v; printf("\"%s\": %u%s\n", k, c.u, last ? "" : ","); }
int main() {
    printf("{\n");
    printf("\"hash32\": [");
    unsigned xs[] = {0u, 1u, 2u, 0xBA5EBA11u, 0xFFFFFFFFu, 123456789u};
    for (int i = 0; i < 6; ++i) printf("[%u, %u]%s", xs[i], MathUtil::hash32(xs[i]), i < 5 ? ", " : "");
    printf("],\n\"pcg\": [");
    UniformSampler s(MathUtil::hash32(0xBA5EBA11u));
    for (int i = 0; i < 8; ++i) printf("%u%s", s.nextI(), i < 7 ? ", " : "");
    printf("],\n\"pcg_seed\": %u,\n\"sobol\": [", MathUtil::hash32(0xBA5EBA11u));
    unsigned idx[] = {0u, 1u, 2u, 3u, 255u, 256u, 1023u, 65535u, 0x12345678u, 0xFFFFFFFFu};
    unsigned dims[] = {0u, 1u, 2u, 7u, 100u, 1023u};
    bool first = true;
    for (unsigned i : idx) for (unsigned d : dims) { printf("%s[%u, %u, %u, %u]", first ? "" : ", ", i, d, 0x9E3779B9u, sobol::sample(i, d, 0x9E3779B9u)); first = false; }
    printf("],\n\"normalized_uint\": [");
    for (int i = 0; i < 6; ++i) { union { float f; unsigned u; } c; c.f = BitManip::normalizedUint(xs[i]); printf("[%u, %u]%s", xs[i], c.u, i < 5 ? ", " : ""); }
    printf("],\n");
    Vec3f ch = SampleWarp::cosineHemisphere(Vec2f(0.3f, 0.7f));
    pf("cos_hemi_x", ch.x()); pf("cos_hemi_y", ch.y()); pf("cos_hemi_z", ch.z());
    pf("dielectric_1.5_0.3", Fresnel::dielectricReflectance(1.0f/1.5f, 0.3f));
    pf("dielectric_1.5_m0.3", Fresnel::dielectricReflectance(1.0f/1.5f, -0.3f));
    pf("conductor_cu_r_0.4", Fresnel::conductorReflectance(0.200438f, 3.91295f, 0.4f));
    pf("diffuse_fresnel_1.5", Fresnel::computeDiffuseFresnel(1.5f, 1000000));
    pf("diffuse_fresnel_1.4", Fresnel::computeDiffuseFresnel(1.4f, 1000000));
    pf("power_heuristic", SampleWarp::powerHeuristic(0.3f, 1.7f));
    TangentFrame tf(Vec3f(0.36f, -0.48f, 0.8f));
    pf("frame_tx", tf.tangent.x()); pf("frame_ty", tf.tangent.y()); pf("frame_tz", tf.tangent.z());
    pf("frame_bx", tf.bitangent.x()); pf("frame_by", tf.bitangent.y()); pf("frame_bz", tf.bitangent.z());
    pf("ggx_D", Microfacet::D(Microfacet::Distribution("ggx"), 0.25f, Vec3f(0.1f, 0.2f, 0.9746794f)));
    pf("beckmann_G1", Microfacet::G1(Microfacet::Distribution("beckmann"), 0.3f, Vec3f(0.6f, 0.0f, 0.8f), Vec3f(0.0f, 0.0f, 1.0f)), true);
    printf("}\n");
}
'''


def make_kat():
    d = tempfile.mkdtemp()
    src = os.path.join(d, "kat.cpp")
    open(src, "w").write(KAT_CPP)
    exe = os.path.join(d, "kat")
    objs = [os.path.join(ROOT, "oracle", "_ref", "obj", "tp", "sobol", "sobol.o")]
    core = os.path.join(ROOT, "oracle", "_ref", "obj", "core")
    # StringableEnum tables for Microfacet::Distribution live in bsdfs/Microfacet.cpp
    objs += [os.path.join(core, "bsdfs", "Microfacet.o")]
    cmd = ["g++", "-std=c++11", "-O2", "-march=core2", "-mno-fma", "-DCONSTEXPR=constexpr", "-I" + REF + "/src/core",
           "-I" + REF + "/src/thirdparty", "-I" + REF + "/src", src] + objs + ["-o", exe]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        # fall back to linking the whole core archive-free object set
        print(r.stdout[-3000:])
        raise SystemExit("KAT program failed to build")
    out = subprocess.check_output([exe], text=True)
    json.loads(out)
    open(os.path.join(HERE, "kat.json"), "w").write(out)
    shutil.rmtree(d)


KAT_CURVES_CPP = r"""
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <memory>
#include <new>
#include <vector>
#include "bsdfs/HairBcsdf.hpp"
#include "primitives/Curves.hpp"
#include "primitives/IntersectionInfo.hpp"
#include "primitives/IntersectionTemporary.hpp"
#include "samplerecords/SurfaceScatterEvent.hpp"
#include "sampling/SobolPathSampler.hpp"
#include "math/TangentFrame.hpp"
#include "math/Ray.hpp"
using namespace Tungsten;
static unsigned bits(float v) { union { float f; unsigned u; } c; c.f = v; return c.u; }
struct CurveIsect { uint32 curveP0; float t; Vec2f uv; float w; };      // mirror of the struct private to Curves.cpp:27-33
int main() {
    // ---- HairBcsdf with its constructor defaults (scale_angle 2, melanin 0.5 / 0.25, roughness 0.1)
    HairBcsdf hair;
    hair.prepareForRender();
    IntersectionInfo info;
    printf("{\n\"hair\": [");
    for (int k = 0; k < 48; ++k) {
        float a = 0.37f*k, b = 1.13f*k + 0.5f;
        Vec3f wi(std::cos(a)*std::cos(0.61f*k), std::sin(0.61f*k)*0.9f, std::sin(a)*std::cos(0.61f*k));
        Vec3f wo(std::cos(b)*std::cos(0.23f*k + 1.0f), std::sin(0.23f*k + 1.0f)*0.95f, std::sin(b)*std::cos(0.23f*k + 1.0f));
        wi.normalize(); wo.normalize();
        SurfaceScatterEvent ev(&info, nullptr, TangentFrame(Vec3f(0.0f, 0.0f, 1.0f)), wi, BsdfLobes::AllLobes, false);
        ev.wo = wo;
        Vec3f f = hair.eval(ev);
        float pdf = hair.pdf(ev);
        printf("%s[%u, %u, %u, %u, %u, %u, %u, %u, %u, %u]", k ? ", " : "", bits(wi.x()), bits(wi.y()), bits(wi.z()), bits(wo.x()), bits(wo.y()),
               bits(wo.z()), bits(f.x()), bits(f.y()), bits(f.z()), bits(pdf));
    }
    // ---- HairBcsdf::sample through the reference's SobolPathSampler (4 Sobol dimensions per draw)
    printf("],\n\"hair_sample_seed\": %u,\n\"hair_samples\": [", 0x0BADC0DEu);
    SobolPathSampler sampler(0x0BADC0DEu);
    for (int k = 0; k < 48; ++k) {
        float a = 0.37f*k;
        Vec3f wi(std::cos(a)*std::cos(0.61f*k), std::sin(0.61f*k)*0.9f, std::sin(a)*std::cos(0.61f*k));
        wi.normalize();
        sampler.startPath(uint32(k), 3);
        SurfaceScatterEvent ev(&info, &sampler, TangentFrame(Vec3f(0.0f, 0.0f, 1.0f)), wi, BsdfLobes::AllLobes, false);
        bool ok = hair.sample(ev);
        printf("%s[%u, %u, %u, %d, %u, %u, %u, %u, %u, %u, %u]", k ? ", " : "", bits(wi.x()), bits(wi.y()), bits(wi.z()), ok ? 1 : 0,
               bits(ev.wo.x()), bits(ev.wo.y()), bits(ev.wo.z()), bits(ev.weight.x()), bits(ev.weight.y()), bits(ev.weight.z()), bits(ev.pdf));
    }
    // ---- Curves::intersect (half_cylinder) on 6 curly strands x 9 nodes
    std::vector<uint32> ends; std::vector<Vec4f> nodes;
    for (int c = 0; c < 6; ++c) {
        for (int i = 0; i < 9; ++i) {
            float s = i/8.0f, ang = 5.0f*s + c;
            nodes.emplace_back(0.4f*c - 1.0f + 0.15f*std::cos(ang), 1.0f - 1.8f*s, 0.15f*std::sin(ang) + 0.05f*c, 0.02f + 0.004f*((c + i) % 3));
        }
        ends.push_back(uint32(nodes.size()));
    }
    printf("],\n\"nodes\": [");
    for (size_t i = 0; i < nodes.size(); ++i) printf("%s[%u, %u, %u, %u]", i ? ", " : "", bits(nodes[i].x()), bits(nodes[i].y()), bits(nodes[i].z()), bits(nodes[i].w()));
    printf("],\n\"ends\": [");
    for (size_t i = 0; i < ends.size(); ++i) printf("%s%u", i ? ", " : "", ends[i]);
    std::shared_ptr<Bsdf> bsdf = std::make_shared<HairBcsdf>();
    // this constructor leaves Curves::_subsample uninitialised (Curves.cpp:278-291); zeroed storage makes it 0 = keep every curve
    void *mem = calloc(1, sizeof(Curves));
    Curves &curves = *new (mem) Curves(ends, nodes, bsdf, "kat");
    curves.prepareForRender();
    printf("],\n\"rays\": [");
    for (int k = 0; k < 400; ++k) {
        Vec3f o(-2.0f + 0.01f*k, 1.5f - 0.007f*k, 2.5f + 0.3f*std::sin(0.7f*k));
        // aim near the curve: a quadratic B-spline segment starts at the midpoint of its first two nodes
        int c = k % 6, i = (k/6) % 8;
        Vec3f mid = (nodes[c*9 + i].xyz() + nodes[c*9 + i + 1].xyz())*0.5f;
        Vec3f tgt = mid + Vec3f(0.03f*std::sin(1.3f*k), 0.02f*std::cos(0.9f*k), 0.0f);
        Vec3f d = (tgt - o).normalized();
        Ray ray(o, d, 1e-4f);
        IntersectionTemporary tmp;
        bool hit = curves.intersect(ray, tmp);
        const CurveIsect *is = tmp.as<CurveIsect>();
        printf("%s[%u, %u, %u, %u, %u, %u, %d, %u, %u, %u, %u, %u]", k ? ", " : "", bits(o.x()), bits(o.y()), bits(o.z()), bits(d.x()), bits(d.y()), bits(d.z()),
               hit ? 1 : 0, hit ? bits(ray.farT()) : 0u, hit ? is->curveP0 : 0u, hit ? bits(is->uv.x()) : 0u, hit ? bits(is->uv.y()) : 0u, hit ? bits(is->w) : 0u);
    }
    printf("]\n}\n");
}
"""


KAT_BSDF_CPP = r"""
#include <cstdio>
#include <cmath>
#include <memory>
#include <vector>
#include "bsdfs/LambertBsdf.hpp"
#include "bsdfs/RoughConductorBsdf.hpp"
#include "bsdfs/RoughDielectricBsdf.hpp"
#include "bsdfs/PlasticBsdf.hpp"
#include "bsdfs/RoughPlasticBsdf.hpp"
#include "bsdfs/SmoothCoatBsdf.hpp"
#include "bsdfs/RoughCoatBsdf.hpp"
#include "bsdfs/MirrorBsdf.hpp"
#include "bsdfs/ConductorBsdf.hpp"
#include "bsdfs/DielectricBsdf.hpp"
#include "textures/ConstantTexture.hpp"
#include "primitives/IntersectionInfo.hpp"
#include "samplerecords/SurfaceScatterEvent.hpp"
#include "sampling/SobolPathSampler.hpp"
#include "math/TangentFrame.hpp"
using namespace Tungsten;
static unsigned bits(float v) { union { float f; unsigned u; } c; c.f = v; return c.u; }
static unsigned lobe_mask(BsdfLobes l) {       // BsdfLobes keeps its bits private: rebuild the mask (bsdfs/BsdfLobes.hpp:13-34)
    unsigned m = 0;
    const BsdfLobes::Lobe all[] = {BsdfLobes::GlossyReflectionLobe, BsdfLobes::GlossyTransmissionLobe, BsdfLobes::DiffuseReflectionLobe,
        BsdfLobes::DiffuseTransmissionLobe, BsdfLobes::SpecularReflectionLobe, BsdfLobes::SpecularTransmissionLobe};
    for (int i = 0; i < 6; ++i) if (l.test(BsdfLobes(all[i]))) m |= 1u << i;
    return m;
}
int main() {
    std::vector<std::shared_ptr<Bsdf>> list;
    { auto b = std::make_shared<LambertBsdf>(); b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.7f, 0.5f, 0.3f))); list.push_back(b); }
    { auto b = std::make_shared<RoughConductorBsdf>(); list.push_back(b); }
    { auto b = std::make_shared<RoughConductorBsdf>(); b->setDistributionName("beckmann"); b->setRoughness(std::make_shared<ConstantTexture>(0.3f));
      b->setEta(Vec3f(0.143f, 0.375f, 1.442f)); b->setK(Vec3f(3.98f, 2.39f, 1.6f)); list.push_back(b); }
    { auto b = std::make_shared<RoughConductorBsdf>(); b->setDistributionName("phong"); b->setRoughness(std::make_shared<ConstantTexture>(0.2f)); list.push_back(b); }
    { auto b = std::make_shared<RoughDielectricBsdf>(); list.push_back(b); }
    { auto b = std::make_shared<RoughDielectricBsdf>(); b->setDistributionName("beckmann"); b->setRoughness(std::make_shared<ConstantTexture>(0.25f)); b->setIor(1.33f); list.push_back(b); }
    { auto b = std::make_shared<PlasticBsdf>(); b->setIor(1.5f); b->setThickness(2.0f); b->setSigmaA(Vec3f(0.1f, 0.2f, 0.3f));
      b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.2f, 0.4f, 0.8f))); list.push_back(b); }
    { auto b = std::make_shared<RoughPlasticBsdf>(); b->setDistributionName("beckmann"); b->setRoughness(std::make_shared<ConstantTexture>(0.3f)); b->setIor(1.4f);
      b->setSigmaA(Vec3f(0.1f, 0.2f, 0.3f)); b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.8f, 0.3f, 0.2f))); list.push_back(b); }
    { auto sub = std::make_shared<RoughConductorBsdf>(); sub->setDistributionName("beckmann");
      auto b = std::make_shared<SmoothCoatBsdf>(); b->setIor(1.7f); b->setThickness(5.0f); b->setSigmaA(Vec3f(0.1f, 0.2f, 0.5f)); b->setSubstrate(sub); list.push_back(b); }
    // the Dirac lobes (appended: the serial PCG stream of the draws above is unchanged)
    { auto b = std::make_shared<MirrorBsdf>(); b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.9f, 0.8f, 0.7f))); list.push_back(b); }
    { auto b = std::make_shared<ConductorBsdf>(); list.push_back(b); }
    { auto b = std::make_shared<ConductorBsdf>(); b->setEta(Vec3f(0.143f, 0.375f, 1.442f)); b->setK(Vec3f(3.98f, 2.39f, 1.6f));
      b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.95f, 0.9f, 0.85f))); list.push_back(b); }
    { auto b = std::make_shared<DielectricBsdf>(); list.push_back(b); }
    { auto b = std::make_shared<DielectricBsdf>(1.33f); b->setEnableTransmission(false); b->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.8f, 0.9f, 1.0f))); list.push_back(b); }
    // RoughCoatBsdf (appended, see above): constructor defaults; Beckmann coat with absorption over Lambert; GGX coat over plastic
    { auto b = std::make_shared<RoughCoatBsdf>(); list.push_back(b); }
    { auto sub = std::make_shared<LambertBsdf>(); sub->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.6f, 0.3f, 0.2f)));
      auto b = std::make_shared<RoughCoatBsdf>(); b->setDistributionName("beckmann"); b->setRoughness(std::make_shared<ConstantTexture>(0.3f)); b->setIor(1.5f);
      b->setThickness(2.0f); b->setSigmaA(Vec3f(0.2f, 0.1f, 0.4f)); b->setSubstrate(sub); list.push_back(b); }
    // (a substrate taken from the scene's bsdf list by name is prepared by TraceableScene, TraceableScene.hpp:76-77; an INLINE
    //  substrate object never is -- Scene::fetchObject only instantiates it -- which leaves PlasticBsdf's derived members unset)
    { auto sub = std::make_shared<PlasticBsdf>(); sub->setAlbedo(std::make_shared<ConstantTexture>(Vec3f(0.2f, 0.5f, 0.7f))); sub->prepareForRender();
      auto b = std::make_shared<RoughCoatBsdf>(); b->setRoughness(std::make_shared<ConstantTexture>(0.15f)); b->setIor(1.6f); b->setSubstrate(sub); list.push_back(b); }
    IntersectionInfo info; info.uv = Vec2f(0.3f, 0.4f);
    printf("{\n\"bsdfs\": [");
    for (size_t n = 0; n < list.size(); ++n) {
        list[n]->prepareForRender();
        printf("%s[", n ? ",\n" : "");
        for (int k = 0; k < 40; ++k) {
            float a = 0.37f*k + 0.1f*n, b = 1.13f*k + 0.5f;
            float zi = 0.05f + 0.9f*std::fabs(std::sin(0.61f*k + 0.3f)), zo = std::sin(0.23f*k + 1.0f);      // wi above, wo on both sides
            if (k % 5 == 0) zi = -zi;                                                                            // and a few wi from below
            Vec3f wi(std::cos(a)*std::sqrt(1.0f - zi*zi), std::sin(a)*std::sqrt(1.0f - zi*zi), zi);
            Vec3f wo(std::cos(b)*std::sqrt(1.0f - zo*zo), std::sin(b)*std::sqrt(1.0f - zo*zo), zo);
            if (k % 7 == 3) wo = Vec3f(-wi.x(), -wi.y(), wi.z());                                                // exact mirror direction
            SurfaceScatterEvent ev(&info, nullptr, TangentFrame(Vec3f(0.0f, 0.0f, 1.0f)), wi, BsdfLobes::AllLobes, false);
            ev.wo = wo;
            Vec3f f = list[n]->eval(ev);
            float pdf = list[n]->pdf(ev);
            printf("%s[%u, %u, %u, %u, %u, %u, %u, %u, %u, %u]", k ? ", " : "", bits(wi.x()), bits(wi.y()), bits(wi.z()), bits(wo.x()), bits(wo.y()),
                   bits(wo.z()), bits(f.x()), bits(f.y()), bits(f.z()), bits(pdf));
        }
        printf("]");
    }
    // ---- sample(): the reference's own SobolPathSampler (stock header: ONE supplemental PCG stream for the whole run),
    //      path (pixel k, sample 7) per draw; output success, wo, weight, pdf, sampled lobe mask
    printf("],\n\"sample_seed\": %u,\n\"samples\": [", 0x5EED1234u);
    SobolPathSampler sampler(0x5EED1234u);
    for (size_t n = 0; n < list.size(); ++n) {
        printf("%s[", n ? ",\n" : "");
        for (int k = 0; k < 40; ++k) {
            float a = 0.37f*k + 0.1f*n;
            float zi = 0.05f + 0.9f*std::fabs(std::sin(0.61f*k + 0.3f));
            if (k % 5 == 0) zi = -zi;
            Vec3f wi(std::cos(a)*std::sqrt(1.0f - zi*zi), std::sin(a)*std::sqrt(1.0f - zi*zi), zi);
            sampler.startPath(uint32(k), 7);
            SurfaceScatterEvent ev(&info, &sampler, TangentFrame(Vec3f(0.0f, 0.0f, 1.0f)), wi, BsdfLobes::AllLobes, false);
            bool ok = list[n]->sample(ev);
            // eval()/pdf() at the sampled direction (all lobes requested): exact mirror / refraction directions for the Dirac lobes
            Vec3f fs(0.0f); float ps = 0.0f;
            if (ok) { SurfaceScatterEvent e2(&info, nullptr, TangentFrame(Vec3f(0.0f, 0.0f, 1.0f)), wi, BsdfLobes::AllLobes, false); e2.wo = ev.wo; fs = list[n]->eval(e2); ps = list[n]->pdf(e2); }
            printf("%s[%u, %u, %u, %d, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u]", k ? ", " : "", bits(wi.x()), bits(wi.y()), bits(wi.z()), ok ? 1 : 0,
                   ok ? bits(ev.wo.x()) : 0u, ok ? bits(ev.wo.y()) : 0u, ok ? bits(ev.wo.z()) : 0u, ok ? bits(ev.weight.x()) : 0u,
                   ok ? bits(ev.weight.y()) : 0u, ok ? bits(ev.weight.z()) : 0u, ok ? bits(ev.pdf) : 0u, ok ? lobe_mask(ev.sampledLobe) : 0u,
                   bits(fs.x()), bits(fs.y()), bits(fs.z()), bits(ps));
        }
        printf("]");
    }
    printf("]\n}\n");
}
"""


def _build_and_run_kat(source, name, out_json, args=()):
    import glob
    d = tempfile.mkdtemp()
    src = os.path.join(d, name + ".cpp")
    open(src, "w").write(source)
    exe = os.path.join(d, name)
    obj = os.path.join(ROOT, "oracle", "_ref", "obj")
    objs = [o for o in glob.glob(os.path.join(obj, "**", "*.o"), recursive=True)
            if not o.endswith("tungsten_main.o") and os.sep + "pathseed" + os.sep not in o]
    cmd = ["/opt/gcc/bin/g++", "-std=c++11", "-O2", "-march=core2", "-mssse3", "-mno-fma", "-DCONSTEXPR=constexpr", "-DRAPIDJSON_HAS_STDSTRING=1",
           "-I" + REF + "/src/core", "-I" + REF + "/src/thirdparty", "-I" + REF + "/src/thirdparty/embree/include", "-I" + REF + "/src", "-w", src] + objs + \
          ["-o", exe, "-lpthread", "-ldl"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout[-3000:])
        raise SystemExit(name + ": KAT program failed to build")
    out = subprocess.check_output([exe] + list(args), text=True)
    json.loads(out)
    open(os.path.join(HERE, out_json), "w").write(out)
    shutil.rmtree(d)


def make_kat_bsdfs():
    """Known answers of eval()/pdf() of the reference's own BSDF classes (nine parameterisations) -> kat_bsdfs.json."""
    _build_and_run_kat(KAT_BSDF_CPP, "kat_bsdfs", "kat_bsdfs.json")


KAT_LIGHTS_CPP = r"""
#include <cstdio>
#include <cstdlib>
#include <cmath>
#include <memory>
#include <vector>
#include "primitives/Quad.hpp"
#include "primitives/TriangleMesh.hpp"
#include "primitives/InfiniteSphere.hpp"
#include "primitives/EmbreeUtil.hpp"
#include "primitives/IntersectionInfo.hpp"
#include "primitives/IntersectionTemporary.hpp"
#include "samplerecords/LightSample.hpp"
#include "sampling/SobolPathSampler.hpp"
#include "textures/ConstantTexture.hpp"
#include "textures/BitmapTexture.hpp"
#include "bsdfs/LambertBsdf.hpp"
#include "math/Ray.hpp"
using namespace Tungsten;
static unsigned bits(float v) { union { float f; unsigned u; } c; c.f = v; return c.u; }
// sampleDirect from point p, then the light's own intersect + intersectionInfo + directPdf + evalDirect along the sampled
// direction (what TraceBase::lightSample / attenuatedEmission / bsdfSample use), one Sobol path per draw
static void probe(Primitive &light, SobolPathSampler &sampler, int n, int sampleIndex) {
    for (int k = 0; k < n; ++k) {
        Vec3f p(-0.8f + 0.07f*k, 0.9f + 0.05f*(k % 7), 0.6f - 0.04f*k);
        sampler.startPath(uint32(k), uint32(sampleIndex));
        LightSample ls;
        bool ok = light.sampleDirect(0, p, sampler, ls);
        unsigned hit = 0; float pdf2 = 0.0f; Vec3f em(0.0f); float t = 0.0f;
        if (ok) {
            Ray ray(p, ls.d, 5e-4f);
            IntersectionTemporary data; IntersectionInfo info;
            if (light.intersect(ray, data)) {
                hit = 1; t = ray.farT();
                info.p = ray.pos() + ray.dir()*ray.farT(); info.w = ray.dir(); info.epsilon = 5e-4f;
                light.intersectionInfo(data, info);
                pdf2 = light.directPdf(0, data, info, p);
                em = light.evalDirect(data, info);
            }
        }
        printf("%s[%u, %u, %u, %d, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u, %u]", k ? ", " : "", bits(p.x()), bits(p.y()), bits(p.z()), ok ? 1 : 0,
               bits(ok ? ls.d.x() : 0.0f), bits(ok ? ls.d.y() : 0.0f), bits(ok ? ls.d.z() : 0.0f), bits(ok ? ls.dist : 0.0f), bits(ok ? ls.pdf : 0.0f),
               hit, bits(t), bits(pdf2), bits(em.x()), bits(em.y()), bits(em.z()));
    }
}
int main() {
    const TraceableScene *noScene = nullptr;                 // makeSamplable of quads and meshes ignores its scene argument
    EmbreeUtil::initDevice();                                 // as the renderer does at start-up (src/tungsten/Shared.hpp:165)
    std::shared_ptr<Bsdf> bsdf = std::make_shared<LambertBsdf>();
    SobolPathSampler sampler(0xC0FFEE11u);
    printf("{\n\"seed\": %u,\n", 0xC0FFEE11u);
    // ---- quad light, identity orientation (normal +y), 1.5 x 1 at y = 0
    Quad quad;
    quad.setTransform(Mat4f::translate(Vec3f(0.1f, 0.0f, -0.2f))*Mat4f::scale(Vec3f(1.5f, 1.0f, 1.0f)));
    quad.setEmission(std::make_shared<ConstantTexture>(Vec3f(3.0f, 2.0f, 1.0f)));
    quad.prepareForRender();
    quad.makeSamplable(*noScene, 0);
    printf("\"quad\": ["); probe(quad, sampler, 40, 2); printf("],\n");
    // ---- mesh light: 5 triangles of different areas facing up / tilted
    std::vector<Vertex> verts = {Vertex(Vec3f(-1.0f, 0.0f, -1.0f)), Vertex(Vec3f(1.0f, 0.0f, -1.0f)), Vertex(Vec3f(1.0f, 0.1f, 1.0f)), Vertex(Vec3f(-1.0f, 0.0f, 1.0f)),
                                 Vertex(Vec3f(0.0f, 0.4f, 0.0f)), Vertex(Vec3f(2.0f, 0.3f, 0.5f))};
    std::vector<TriangleI> tris = {TriangleI(0, 2, 1, 0), TriangleI(0, 3, 2, 0), TriangleI(0, 4, 1, 0), TriangleI(1, 5, 2, 0), TriangleI(3, 4, 2, 0)};
    TriangleMesh mesh(verts, tris, bsdf, "kat", false, false);
    mesh.setTransform(Mat4f::translate(Vec3f(0.0f, -0.3f, 0.0f)));
    mesh.setEmission(std::make_shared<ConstantTexture>(Vec3f(1.0f, 4.0f, 2.0f)));
    mesh.prepareForRender();
    mesh.makeSamplable(*noScene, 0);
    printf("\"mesh\": ["); probe(mesh, sampler, 40, 3); printf("],\n");
    // ---- environment sphere with a 32x16 RGB bitmap (exactly representable texels), importance sampled
    const int W = 32, H = 16;
    Vec3f *texels = new Vec3f[W*H];
    for (int y = 0; y < H; ++y) for (int x = 0; x < W; ++x)
        texels[x + y*W] = Vec3f(1.0f + float((x*7 + y*3) % 11), 0.5f + float((x*5 + y) % 7), 0.25f*float((x + y) % 5));
    auto tex = std::make_shared<BitmapTexture>(texels, W, H, BitmapTexture::TexelType::RGB_HDR, true, false);
    InfiniteSphere sphere;
    sphere.setEmission(tex);
    sphere.prepareForRender();
    tex->makeSamplable(MAP_SPHERICAL);                       // what InfiniteSphere::makeSamplable does besides caching the scene bounds
    printf("\"env\": ["); probe(sphere, sampler, 48, 4); printf("]\n}\n");
}
"""


KAT_INSTANCE_CPP = r'''
// Instance transforms through the reference's own classes: Instance::fromJson (Instance.cpp:80-86) turns an instance matrix into
// (extractTranslationVec, QuaternionF::fromMatrix(extractRotation)); prepareForRender (:392-400) composes it with the
// primitive's transform (_transform*pos, rot*instanceRot); intersectionInfo (:325-334) maps master-space points / normals to
// the world with pos + rot*p, rot*n.
#include <cstdio>
#include "math/Mat4f.hpp"
#include "math/Quaternion.hpp"
#include "sampling/UniformSampler.hpp"
using namespace Tungsten;
static unsigned bits(float v) { union { float f; unsigned u; } c; c.f = v; return c.u; }
static void pv(const char *k, const float *v, int n, bool last = false) { printf("\"%s\": [", k); for (int i = 0; i < n; ++i) printf("%u%s", bits(v[i]), i + 1 < n ? ", " : ""); printf("]%s", last ? "" : ", "); }
int main() {
    UniformSampler rnd(0x5EED1234u);
    printf("{\"cases\": [\n");
    const int N = 32;
    for (int c = 0; c < N; ++c) {
        Vec3f ang(rnd.next1D()*360.0f - 180.0f, rnd.next1D()*360.0f - 180.0f, rnd.next1D()*360.0f - 180.0f);
        Vec3f ang2(rnd.next1D()*360.0f - 180.0f, rnd.next1D()*360.0f - 180.0f, rnd.next1D()*360.0f - 180.0f);
        if (c < 4) { ang = Vec3f(0.0f, 90.0f*c, 0.0f); ang2 = Vec3f(180.0f, 0.0f, 90.0f*c); }          // exercise every fromMatrix branch
        Vec3f tr(rnd.next1D()*40.0f - 20.0f, rnd.next1D()*4.0f, rnd.next1D()*40.0f - 20.0f);
        Vec3f tr2(rnd.next1D()*10.0f - 5.0f, rnd.next1D()*2.0f, rnd.next1D()*10.0f - 5.0f);
        float sc = c % 3 == 0 ? 1.0f : 0.5f + rnd.next1D();
        Mat4f inst = Mat4f::translate(tr)*Mat4f::rotYXZ(ang);                       // one entry of "instances"
        Mat4f prim = Mat4f::translate(tr2)*Mat4f::rotYXZ(ang2)*Mat4f::scale(Vec3f(sc));   // the Instance primitive's own transform
        Vec3f ipos = inst.extractTranslationVec();
        QuaternionF irot = QuaternionF::fromMatrix(inst.extractRotation());
        QuaternionF prot = QuaternionF::fromMatrix(prim.extractRotation());
        Vec3f wpos = prim*ipos;
        QuaternionF wrot = prot*irot;
        float m1[16], m2[16];
        for (int i = 0; i < 16; ++i) { m1[i] = inst[i]; m2[i] = prim[i]; }
        printf("{"); pv("inst", m1, 16); pv("prim", m2, 16);
        float q[4] = {irot[0], irot[1], irot[2], irot[3]}; pv("irot", q, 4);
        float qw[4] = {wrot[0], wrot[1], wrot[2], wrot[3]}; pv("wrot", qw, 4);
        float wp[3] = {wpos.x(), wpos.y(), wpos.z()}; pv("wpos", wp, 3);
        float pts[4*3], outp[4*3], outn[4*3];
        for (int k = 0; k < 4; ++k) {
            Vec3f p(rnd.next1D()*2.0f - 1.0f, rnd.next1D()*3.0f, rnd.next1D()*2.0f - 1.0f);
            Vec3f w = wpos + wrot*p, n = wrot*p;
            for (int a = 0; a < 3; ++a) { pts[3*k + a] = p[a]; outp[3*k + a] = w[a]; outn[3*k + a] = n[a]; }
        }
        pv("p", pts, 12); pv("world_p", outp, 12); pv("world_n", outn, 12, true);
        printf("}%s\n", c + 1 < N ? "," : "");
    }
    printf("]}\n");
}
'''


def make_kat_instances():
    """Instance transforms (quaternion + translation) through the reference's Mat4f / QuaternionF -> kat_instances.json."""
    _build_and_run_kat(KAT_INSTANCE_CPP, "kat_instances", "kat_instances.json")


SKY_DUMP_CPP = r'''
// Dumps the image Skydome::prepareForRender computes (Hosek-Wilkie model, thirdparty/skylight) for the first skydome of a scene
// file: 512 x 256 RGB float32, top row first, raw.
#include <cstdio>
#include <memory>
#include "io/Scene.hpp"
#include "primitives/Skydome.hpp"
#include "textures/BitmapTexture.hpp"
#include "thread/ThreadUtils.hpp"
using namespace Tungsten;
int main(int argc, char **argv) {
    ThreadUtils::startThreads(1);
    std::unique_ptr<Scene> scene(Scene::load(Path(argv[1])));
    for (const std::shared_ptr<Primitive> &p : scene->primitives()) {
        Skydome *sky = dynamic_cast<Skydome *>(p.get());
        if (!sky) continue;
        sky->prepareForRender();
        BitmapTexture *b = dynamic_cast<BitmapTexture *>(sky->emission().get());
        std::unique_ptr<Texture> owner(b->clone());
        BitmapTexture *nearest = static_cast<BitmapTexture *>(owner.get());
        nearest->setLinear(false);
        FILE *f = fopen(argv[2], "wb");
        for (int y = 0; y < b->h(); ++y) for (int x = 0; x < b->w(); ++x) {
            Vec3f c = (*nearest)[Vec2f((x + 0.5f)/b->w(), 1.0f - (y + 0.5f)/b->h())];
            float v[3] = {c.x(), c.y(), c.z()};
            fwrite(v, 4, 3, f);
        }
        fclose(f);
        printf("%d %d\n", b->w(), b->h());
        return 0;
    }
    return 1;
}
'''


def dump_sky_image(scene_json, out_pfm):
    """Skydome::prepareForRender of the scene's skydome, through the reference's own classes -> PFM (the flattener's "sky_image")."""
    import glob
    import numpy as np
    from tungsten_b200 import scene as S
    d = tempfile.mkdtemp()
    src = os.path.join(d, "skydump.cpp"); open(src, "w").write(SKY_DUMP_CPP)
    exe = os.path.join(d, "skydump")
    obj = os.path.join(ROOT, "oracle", "_ref", "obj")
    objs = [o for o in glob.glob(os.path.join(obj, "**", "*.o"), recursive=True)
            if not o.endswith("tungsten_main.o") and os.sep + "pathseed" + os.sep not in o]
    cmd = ["/opt/gcc/bin/g++", "-std=c++11", "-O2", "-march=core2", "-mssse3", "-mno-fma", "-DCONSTEXPR=constexpr", "-DRAPIDJSON_HAS_STDSTRING=1",
           "-I" + REF + "/src/core", "-I" + REF + "/src/thirdparty", "-I" + REF + "/src/thirdparty/embree/include", "-I" + REF + "/src", "-w", src] + objs + \
          ["-o", exe, "-lpthread", "-ldl"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout[-3000:]); raise SystemExit("sky dump program failed to build")
    raw = os.path.join(d, "sky.bin")
    w, h = [int(x) for x in subprocess.check_output([exe, os.path.abspath(scene_json), raw], text=True).split()]
    img = np.fromfile(raw, dtype=np.float32).reshape(h, w, 3)
    S.save_pfm(out_pfm, img)
    shutil.rmtree(d)
    return img


# Closest hits of the reference's own TraceableScene::intersect (Embree BVH4 + Moeller-Trumbore for meshes, the top-level
# user-geometry BVH for quads / cubes) on a scene loaded by the reference's own Scene::load: SURVEY 7 step 1-iii's "--dump-hits".
KAT_SCENE_HITS_CPP = r"""
#include <cstdio>
#include <cstdlib>
#include <vector>
#include <memory>
#include "io/Scene.hpp"
#include "io/Path.hpp"
#include "renderer/TraceableScene.hpp"
#include "primitives/EmbreeUtil.hpp"
#include "primitives/TriangleMesh.hpp"
#include "primitives/IntersectionInfo.hpp"
#include "primitives/IntersectionTemporary.hpp"
#include "thread/ThreadUtils.hpp"
#include "math/Ray.hpp"
using namespace Tungsten;
static unsigned bits(float v) { union { float f; unsigned u; } c; c.f = v; return c.u; }
struct MeshIntersectionView { Vec3f Ng; float u; float v; int primId; bool backSide; };     // TriangleMesh.cpp:22-29 (private to that file)
int main(int argc, char **argv) {
    EmbreeUtil::initDevice();
    ThreadUtils::startThreads(2);
    std::unique_ptr<Scene> scene(Scene::load(Path(argv[1])));
    scene->loadResources();
    std::unique_ptr<TraceableScene> flat(scene->makeTraceable(0xBA5EBA11u));
    FILE *f = fopen(argv[2], "rb");
    std::vector<float> rays; float buf[8];
    while (fread(buf, 4, 8, f) == 8) rays.insert(rays.end(), buf, buf + 8);
    fclose(f);
    printf("{\"hits\": [");
    size_t n = rays.size()/8;
    for (size_t i = 0; i < n; ++i) {
        const float *r = &rays[8*i];
        Ray ray(Vec3f(r[0], r[1], r[2]), Vec3f(r[3], r[4], r[5]), r[6]);
        IntersectionTemporary data; IntersectionInfo info;
        bool hit = flat->intersect(ray, data, info);
        int prim = -1, tri = -1; unsigned back = 0;
        if (hit) {
            for (size_t k = 0; k < scene->primitives().size(); ++k) if (scene->primitives()[k].get() == info.primitive) prim = int(k);
            if (dynamic_cast<const TriangleMesh *>(info.primitive)) tri = data.as<MeshIntersectionView>()->primId;
            back = info.primitive->hitBackside(data) ? 1u : 0u;
        }
        printf("%s[%d, %d, %u, %u]", i ? ", " : "", prim, tri, hit ? bits(ray.farT()) : 0u, back);
    }
    printf("]}\n");
    return 0;
}
"""


def scene_hit_rays(n=6000, seed=11):
    """The rays of kat_scene_hits.json (tests regenerate them from the seed): origins in the room, uniform directions."""
    import numpy as np
    rng = np.random.RandomState(seed)
    o = rng.uniform(-0.9, 0.9, (n, 3)).astype(np.float32); o[:, 1] = rng.uniform(0.05, 1.9, n).astype(np.float32)
    d = rng.normal(size=(n, 3)); d /= np.linalg.norm(d, axis=1, keepdims=True)
    return np.concatenate([o, d.astype(np.float32), np.full((n, 1), 5e-4, np.float32), np.full((n, 1), np.inf, np.float32)], axis=1).astype(np.float32)


def make_kat_scene_hits():
    rays = scene_hit_rays()
    d = tempfile.mkdtemp()
    rp = os.path.join(d, "rays.bin"); rays.tofile(rp)
    _build_and_run_kat(KAT_SCENE_HITS_CPP, "kat_scene_hits", "kat_scene_hits.json", args=[os.path.join(HERE, "materials", "scene.json"), rp])
    shutil.rmtree(d)


def make_kat_lights():
    """Known answers of sampleDirect / intersect / directPdf / evalDirect of the reference's Quad, TriangleMesh and
    InfiniteSphere(+BitmapTexture importance map) classes -> kat_lights.json."""
    _build_and_run_kat(KAT_LIGHTS_CPP, "kat_lights", "kat_lights.json")


def make_kat_curves():
    """Known answers of HairBcsdf::eval/pdf and Curves::intersect from the reference's own classes -> kat_curves.json."""
    import glob
    d = tempfile.mkdtemp()
    src = os.path.join(d, "kat_curves.cpp")
    open(src, "w").write(KAT_CURVES_CPP)
    exe = os.path.join(d, "kat_curves")
    obj = os.path.join(ROOT, "oracle", "_ref", "obj")
    objs = [o for o in glob.glob(os.path.join(obj, "**", "*.o"), recursive=True)
            if not o.endswith("tungsten_main.o") and os.sep + "pathseed" + os.sep not in o]
    cmd = ["/opt/gcc/bin/g++", "-std=c++11", "-O2", "-march=core2", "-mssse3", "-mno-fma", "-DCONSTEXPR=constexpr", "-DRAPIDJSON_HAS_STDSTRING=1",
           "-I" + REF + "/src/core", "-I" + REF + "/src/thirdparty", "-I" + REF + "/src/thirdparty/embree/include", "-I" + REF + "/src", "-w", src] + objs + \
          ["-o", exe, "-lpthread", "-ldl"]
    r = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if r.returncode != 0:
        print(r.stdout[-3000:])
        raise SystemExit("curve KAT program failed to build")
    out = subprocess.check_output([exe], text=True)
    json.loads(out)
    open(os.path.join(HERE, "kat_curves.json"), "w").write(out)
    shutil.rmtree(d)


def make_scenes(only=None):
    import numpy as np
    from tungsten_b200 import synth
    scenes = {}
    res, spp = (64, 64), 8
    d = os.path.join(HERE, "cornell"); os.makedirs(d, exist_ok=True)
    scenes["cornell"] = synth.write_scene(d, "scene", synth.cornell_box(res=res, spp=spp))
    d = os.path.join(HERE, "cornell_short"); os.makedirs(d, exist_ok=True)
    scenes["cornell_short"] = synth.write_scene(d, "scene", synth.cornell_box(res=res, spp=spp, max_bounces=3, filter_name="gaussian"))
    scenes["cornell_mesh"] = synth.cornell_mesh(os.path.join(HERE, "cornell_mesh"), "scene", subdiv=2, res=res, spp=spp)
    scenes["materials"] = synth.material_room(os.path.join(HERE, "materials"), "scene", res=res, spp=spp, subdiv=2)
    scenes["materials_env"] = synth.material_room(os.path.join(HERE, "materials_env"), "scene", res=res, spp=spp, subdiv=2, env=[0.4, 0.5, 0.7])
    scenes["coat_env"] = synth.materialtest_standin(os.path.join(HERE, "coat_env"), "scene", res=res, spp=spp, subdiv=2, env_res=(64, 32))
    # C4 stand-ins: curves primitive + hair BCSDF (bcsdf_cylinder), and the two other curve modes with ordinary lobes
    scenes["hair"] = synth.hair_scene(os.path.join(HERE, "hair"), "scene", n_curves=400, res=res, spp=spp)
    scenes["hair_dark"] = synth.hair_scene(os.path.join(HERE, "hair_dark"), "scene", n_curves=300, res=res, spp=spp, thickness=0.008,
                                           subsample=0.5, env=None, bsdf={"type": "hair", "roughness": 0.1, "scale_angle": 3, "sigma_a": [0.1, 0.2, 0.5]})
    scenes["curves_lambert"] = synth.hair_scene(os.path.join(HERE, "curves_lambert"), "scene", n_curves=300, res=res, spp=spp, mode="half_cylinder",
                                                bsdf={"type": "lambert", "albedo": [0.6, 0.4, 0.2]}, width=0.02)
    scenes["curves_plastic"] = synth.hair_scene(os.path.join(HERE, "curves_plastic"), "scene", n_curves=300, res=res, spp=spp, mode="cylinder",
                                                bsdf={"type": "rough_plastic", "albedo": [0.6, 0.4, 0.2], "roughness": 0.2}, thickness=0.015,
                                                taper=True, subsample=0.3)
    # 39 samplable lights (36 quads + the ceiling light + 2 mesh lights): chooseLight beyond 16 lights
    scenes["many_lights"] = synth.many_lights(os.path.join(HERE, "many_lights"), "scene", res=res, spp=spp, subdiv=2)
    # 151 analytic primitives, no mesh: from 24 on the library keeps them in BVH leaves instead of its per-ray loop
    scenes["cube_city"] = synth.cube_city(os.path.join(HERE, "cube_city"), "scene", n=12, res=res, spp=spp)
    # RoughCoatBsdf over Lambert / rough conductor / plastic substrates (+ a smooth coat)
    scenes["coats"] = synth.coat_room(os.path.join(HERE, "coats"), "scene", res=res, spp=spp, subdiv=2)
    scenes["dirac"] = synth.dirac_room(os.path.join(HERE, "dirac"), "scene", res=res, spp=spp, subdiv=2)
    # the two emitters of the shipped hair scene: infinite_sphere_cap (sampled sun) + skydome (unsampled sky); min_bounces 1 as shipped
    scenes["hair_sky"] = synth.hair_scene(os.path.join(HERE, "hair_sky"), "scene", n_curves=300, res=res, spp=spp, shipped_lights=True, min_bounces=1)
    # the sky image is zero below the horizon (its lower 126 rows): only the rows above are stored, tests pad the rest
    sky = dump_sky_image(scenes["hair_sky"], os.path.join(tempfile.mkdtemp(), "scene_sky.pfm"))
    from tungsten_b200 import scene as S
    above = np.where(sky.any(axis=(1, 2)))[0]
    assert above[0] == 0 and not sky[above[-1] + 1:].any() and 2*len(sky) == sky.shape[1]
    S.save_pfm(os.path.join(HERE, "hair_sky", "scene_sky_top.pfm"), sky[:above[-1] + 1])
    # adaptive sampling (PathTraceIntegrator::generateWork): three 16-spp steps, the 2nd and 3rd distributed by the blocks' error
    ad = synth.cornell_box(res=res, spp=48)
    ad["renderer"].update(adaptive_sampling=True, spp_step=16)
    d = os.path.join(HERE, "cornell_adaptive"); os.makedirs(d, exist_ok=True)
    scenes["cornell_adaptive"] = synth.write_scene(d, "scene", ad)
    for name, path in scenes.items():
        if only and name not in only:
            continue
        d = os.path.dirname(path)
        for exe, tag in (("tungsten_pathseed", "ref_pathseed"), ("tungsten", "ref_stock")):
            out = tempfile.mkdtemp()
            subprocess.check_call([os.path.join(ROOT, "oracle", "_ref", exe), "-t", "4", "-d", out, path], stdout=subprocess.DEVNULL)
            shutil.copy(os.path.join(out, "out.pfm"), os.path.join(d, tag + ".pfm"))
            shutil.rmtree(out)
        print("golden:", name)


def make_sobol_reference():
    """The direction matrices of the reference's src/thirdparty/sobol/sobol.cpp, as far as the library uses them (first 32
    of 52 bits, 1024 dimensions): their SHA-256 and 256 entries at seeded positions -> sobol_reference.json."""
    import hashlib
    import re
    import numpy as np
    txt = open(os.path.join(REF, "src", "thirdparty", "sobol", "sobol.cpp")).read()
    body = txt[txt.index("matrices[Matrices::num_dimensions"):]
    nums = np.array([int(x, 16) for x in re.findall(r"0x([0-9a-fA-F]+)U", body)], dtype=np.uint64).reshape(1024, 52)[:, :32]
    rng = np.random.RandomState(5)
    at = np.stack([rng.randint(0, 1024, 256), rng.randint(0, 32, 256)], axis=1)
    out = {"sha256": hashlib.sha256(np.ascontiguousarray(nums, dtype="<u4").tobytes()).hexdigest(),
           "entries": [[int(d), int(b), int(nums[d, b])] for d, b in at]}
    json.dump(out, open(os.path.join(HERE, "sobol_reference.json"), "w"))


def _cluster_mesh(verts, tris, cells):
    """Vertex-clustering decimation: one vertex per occupied cell of a `cells`^3 grid over the bounding box (mean position,
    uv and renormalised normal of the vertices it replaces); triangles that collapse or repeat are dropped."""
    import numpy as np
    from tungsten_b200 import scene as S
    lo = verts["pos"].min(axis=0); ext = np.maximum(verts["pos"].max(axis=0) - lo, 1e-6)
    c = np.minimum((((verts["pos"] - lo)/ext)*cells).astype(np.int64), cells - 1)
    _, cell_of, counts = np.unique(c[:, 0]*cells*cells + c[:, 1]*cells + c[:, 2], return_inverse=True, return_counts=True)
    out = np.zeros(len(counts), S.VERTEX_DTYPE)
    for f in ("pos", "normal", "uv"):
        acc = np.zeros((len(counts), out[f].shape[1]), np.float64)
        np.add.at(acc, cell_of, verts[f].astype(np.float64))
        out[f] = acc/counts[:, None]
    out["normal"] /= np.maximum(np.linalg.norm(out["normal"], axis=1, keepdims=True), 1e-12)
    idx = cell_of[np.stack([tris["v0"], tris["v1"], tris["v2"]], axis=1).astype(np.int64)]
    keep = (idx[:, 0] != idx[:, 1]) & (idx[:, 1] != idx[:, 2]) & (idx[:, 0] != idx[:, 2])
    _, first = np.unique(np.sort(idx[keep], axis=1), axis=0, return_index=True)
    sel = np.where(keep)[0][np.sort(first)]
    t = np.zeros(len(sel), S.TRI_DTYPE)
    t["v0"], t["v1"], t["v2"] = idx[sel, 0], idx[sel, 1], idx[sel, 2]
    t["material"] = tris["material"][sel]
    return out, t


def make_shipped_scenes():
    """Shrunk copies of two scenes the reference ships, with the reference binary's renders of them (np.savez_compressed,
    key "img"): tests/test_oracle_golden.py compares the oracle with these.
      materialtest/   data/materialtest: the three meshes decimated by vertex clustering, envmap.hdr box-filtered to 64x32;
                      ref_pathseed.npz = 64x64, 8 spp
      hair_shipped/   data/example-scenes/hair: scene.json as shipped, curl.fiber reduced to 100 of its 10,000 strands (seed 7);
                      ref_pathseed_lights.npz = its curves under an environment sphere + quad light, min_bounces 0;
                      ref_pathseed_lights_nocurves.npz = the same lights without the curves (tells the strands' pixels apart);
                      ref_pathseed.npz = the scene with its own emitters (skydome image: hair_sky/scene_sky_top.pfm, the same dome)
                      all 90x300, 2 spp"""
    import numpy as np
    from tungsten_b200 import scene as S, synth

    def render(d, js, name):
        out = tempfile.mkdtemp()
        p = os.path.join(d, "_render.json"); json.dump(js, open(p, "w"))
        subprocess.check_call([os.path.join(ROOT, "oracle", "_ref", "tungsten_pathseed"), "-t", "8", "-d", out, p], stdout=subprocess.DEVNULL)
        np.savez_compressed(os.path.join(d, name), img=S.load_pfm(os.path.join(out, "out.pfm")))
        os.remove(p); shutil.rmtree(out)

    src = os.path.join(REF, "data", "materialtest")
    d = os.path.join(HERE, "materialtest"); os.makedirs(d, exist_ok=True)
    js = json.load(open(os.path.join(src, "materialtest.json")))
    for p in js["primitives"]:
        if p["type"] == "mesh":
            v, t = _cluster_mesh(*S.load_wo3(os.path.join(src, p["file"])), cells=12)
            S.save_wo3(os.path.join(d, p["file"]), v, t)
    env = S.load_rgbe(os.path.join(src, "envmap.hdr"))
    fy, fx = env.shape[0]//32, env.shape[1]//64
    synth.save_rgbe(os.path.join(d, "envmap.hdr"), env[:32*fy, :64*fx].reshape(32, fy, 64, fx, 3).mean(axis=(1, 3)).astype(np.float32))
    js["camera"]["resolution"] = [64, 64]
    js["renderer"].update(spp=8, spp_step=8, adaptive_sampling=False, stratified_sampler=True, hdr_output_file="out.pfm",
                          output_file="out.png", overwrite_output_files=True)
    json.dump(js, open(os.path.join(d, "scene.json"), "w"), indent=1)
    render(d, js, "ref_pathseed.npz")

    src = os.path.join(REF, "data", "example-scenes", "hair")
    d = os.path.join(HERE, "hair_shipped"); os.makedirs(d, exist_ok=True)
    shutil.copyfile(os.path.join(src, "scene.json"), os.path.join(d, "scene.json"))
    ends, nodes = S.load_fiber(os.path.join(src, "curl.fiber"))
    starts = np.concatenate([[0], ends[:-1]])
    keep = np.sort(np.random.RandomState(7).choice(len(ends), 100, replace=False))
    strands = [nodes[starts[k]:ends[k]] for k in keep]
    S.save_fiber(os.path.join(d, "curl.fiber"), np.cumsum([len(s) for s in strands]).astype(np.uint32), np.concatenate(strands))
    js = json.load(open(os.path.join(d, "scene.json")))
    js["primitives"] = [p for p in js["primitives"] if p["type"] == "curves"] + [
        {"name": "env", "type": "infinite_sphere", "emission": [0.5, 0.6, 0.8], "sample": True},
        {"name": "key", "type": "quad", "emission": [60, 55, 50], "bsdf": {"type": "null"},
         "transform": {"position": [3.0, 9.0, 6.0], "scale": [3, 1, 3], "rotation": [0, 0, 140]}}]
    js["integrator"]["min_bounces"] = 0
    for shipped_lights in (False, True):
        if shipped_lights:
            js = json.load(open(os.path.join(d, "scene.json")))
        js["camera"]["resolution"] = [90, 300]
        js["renderer"].update(spp=2, spp_step=2, adaptive_sampling=False, stratified_sampler=True, hdr_output_file="out.pfm",
                              output_file="out.png", overwrite_output_files=True)
        render(d, js, "ref_pathseed.npz" if shipped_lights else "ref_pathseed_lights.npz")
        if not shipped_lights:
            render(d, dict(js, primitives=[p for p in js["primitives"] if p["type"] != "curves"]), "ref_pathseed_lights_nocurves.npz")


if __name__ == "__main__":
    make_kat()
    make_sobol_reference()
    make_kat_curves()
    make_kat_bsdfs()
    make_kat_lights()
    make_kat_instances()
    make_kat_scene_hits()
    make_scenes()
    make_shipped_scenes()
