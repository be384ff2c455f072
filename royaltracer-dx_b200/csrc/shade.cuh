// shade.cuh — device restatement of the reference's material / BSDF / light-sampling arithmetic
// (shaders/{Common,GGX,BRDF,Sampler,Hit,Reservoir}_v7.hlsl and include/Lambertian_v6.hlsl; file:line cited per function,
// relative to /root/reference/Pathtracer/).  Operation order is fixed (see dmath.cuh); half-precision fields of
// MaterialOptimized / Reservoir_* are honoured (true 16-bit types, rdn/DXRHelper.h:125).
#pragma once
#include "common.cuh"
#include "dmath.cuh"

namespace rtx {

struct ModelRef {               // bindings t2/t1 of the hit-group record (rdn/Renderer.cpp:983-1008)
    const uint8_t* verts;       // stride 28: float3 position, float4 normal_material
    const uint32_t* idx;
    uint32_t mat_offset;        // offset into materialIDs (shaders/Hit_v7.hlsl:16-17)
    uint32_t n_tris;
    // closest-hit attribute records, 80 B = 5 x float4 per triangle in primitive order, derived from (verts, idx) at upload:
    // (p0, n0.x) (p1, n0.y) (p2, n0.z) (n1, -) (n2, -).  ClosestHit reads ONE contiguous record instead of three indices and then three
    // 28-byte vertices scattered over the vertex buffer (2.5 instead of ~7 sectors, and one level less of dependent loads).
    const float4* shade;
};

struct SceneData {              // global root signature (rdn/Renderer.cpp:953-976)
    const ModelRef* models;
    const uint32_t* inst_model; // instance -> model
    const rtx_instance_props* props;        // t3
    const uint32_t* material_ids; uint32_t n_material_ids;   // t4
    const rtx_material* materials; uint32_t n_materials;     // t5
    const rtx_light_triangle* lights;                         // t6 (never empty: a zero light stands in)
    uint32_t cfg_flags, bounces, nee_samples, nee_samples_di;
    uint32_t width, height;
    // world bounds of the instances whose BLAS holds at least a quarter of the largest BLAS's triangles (api.cu rtx_set_instances);
    // heavy_valid = 0: queues are filled from one end only
    float heavy_lo[3], heavy_hi[3]; uint32_t heavy_valid;
};

struct MatOpt {                 // shaders/Common_v7.hlsl:62-66 — every float holds a binary16 value
    f3 Kd; float Pr, Pm;
    f3 Ks; f3 Ke;
    uint32_t mID;
};

struct HitInfo {                // shaders/Common_v7.hlsl:35-46
    f3 hitPosition; uint32_t materialID; f3 hitNormal; uint32_t objID;
};

// OOB StructuredBuffer reads return 0 (SURVEY.md Appendix C.3)
__device__ __forceinline__ void fetch_material_head(const SceneData& S, uint32_t id, float4& kd, float4& ks_ni, float4& ke_pad, float4& pr) {
    if (id < S.n_materials) {
        const float4* m = reinterpret_cast<const float4*>(S.materials + id);
        kd = __ldg(m); ks_ni = __ldg(m + 1); ke_pad = __ldg(m + 2); pr = __ldg(m + 3);
    } else {
        kd = ks_ni = ke_pad = pr = make_float4(0, 0, 0, 0);
    }
}
// Pass_init_di_v7.hlsl:108-111 / Sampler_v7.hlsl:71-82.  ke_full returns the un-rounded Ke (Material, not MaterialOptimized).
__device__ __forceinline__ MatOpt load_matopt(const SceneData& S, uint32_t id, f3* ke_full) {
    float4 kd, ks, ke, pr;
    fetch_material_head(S, id, kd, ks, ke, pr);
    MatOpt o;
    o.Kd = mk3(q16(kd.x), q16(kd.y), q16(kd.z));
    o.Pr = q16(pr.x); o.Pm = q16(pr.y);
    o.Ks = mk3(q16(ks.x), q16(ks.y), q16(ks.z));
    o.Ke = mk3(q16(ke.x), q16(ke.y), q16(ke.z));
    o.mID = id;
    if (ke_full) *ke_full = mk3(ke.x, ke.y, ke.z);
    return o;
}

// shaders/Common_v7.hlsl:119-138
// One out-of-line copy per kernel: the shading stages draw ~20 numbers per bounce, inlined that is ~1200 of k_gi_step's 4000 SASS
// instructions, and the kernel stalls on instruction fetch (ncu: no_instruction 1.65 stall cycles per issue).  k_gi_step 3.78 -> 3.70 ms
// per C2 pass (profiles/r02_s1_stage_times.txt).
static __device__ __noinline__ uint2 tea4(uint2 seed) {
    uint32_t v0 = seed.x, v1 = seed.y, sum = 0u;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        sum += 0x9e3779b9u;
        v0 += ((v1 << 4) + 0xA341316Cu) ^ (v1 + sum) ^ ((v1 >> 5) + 0xC8013EA4u);
        v1 += ((v0 << 4) + 0xAD90777Du) ^ (v0 + sum) ^ ((v0 >> 5) + 0x7E95761Eu);
    }
    return make_uint2(v0, v1);
}
__device__ __forceinline__ float RandomFloat(uint2& seed) {
    seed = tea4(seed);
    return (float)seed.x / 4294967296.0f;
}
// shaders/Pass_init_di_v7.hlsl:63-77, uint(time) := global sample index
__device__ __forceinline__ uint2 init_seed(uint32_t x, uint32_t y, uint32_t pass, uint32_t sample) {
    uint2 s;
    s.x = (y * 73856093u) ^ (x * 19349663u) ^ (pass * 83492791u) ^ (sample * 293803u);
    s.y = (x * 37623481u) ^ (y * 51964263u) ^ (pass * 68250729u) ^ (sample * 423977u);
    return s;
}

// shaders/Common_v7.hlsl:151-160
__device__ __forceinline__ f3 SafeMultiply(float s, f3 v) {
    f3 r = s * v;
    if (any_nan_inf(r)) return mk3(0, 0, 0);
    return r;
}
__device__ __forceinline__ float SafeMultiply1(float s, float v) {
    float r = s * v;
    if (isnan1(r) || isinf1(r)) return 0.0f;
    return r;
}

// ---- shaders/GGX_v7.hlsl
// :1-23
__device__ __forceinline__ float ESS_LUT(const SceneData& S, const MatOpt& mat, float NdotV) {
    NdotV = saturate1(NdotV);
    float thetaIdxF = NdotV * 15.0f;
    int i0 = (int)floorf(thetaIdxF);
    int i1 = min(i0 + 1, 15);
    float w = thetaIdxF - (float)i0;
    float v0 = 0.0f, v1 = 0.0f;
    if (mat.mID < S.n_materials) { v0 = __ldg(&S.materials[mat.mID].LUT[i0]); v1 = __ldg(&S.materials[mat.mID].LUT[i1]); }
    return lerp1(v0, v1, w);
}
// :26-29
__device__ __forceinline__ f3 SchlickFresnel(f3 F0, float cosTheta) {
    float x = fabsf(1.0f - cosTheta);
    float p = (((x * x) * x) * x) * x;
    return saturate3(mk3(F0.x + (1.0f - F0.x) * p, F0.y + (1.0f - F0.y) * p, F0.z + (1.0f - F0.z) * p));
}
// :31-40
template <class M = Ieee>
__device__ __forceinline__ float D_GGX(float NdotH, float roughness, M m = M()) {
    float alpha = roughness * roughness;
    float alpha2 = alpha * alpha;
    float NdotH2 = NdotH * NdotH;
    float denom = (NdotH2 * (alpha2 - 1.0f) + 1.0f);
    return m.div(alpha2, (RTX_PI_REF * denom) * denom);
}
// :43-52
template <class M = Ieee>
__device__ __forceinline__ float G2_SmithGGX(float NdotV, float NdotL, float alpha, M m = M()) {
    float alpha2 = alpha * alpha;
    float denomA = NdotV * m.sqrt(alpha2 + ((1.0f - alpha2) * NdotL) * NdotL);
    float denomB = NdotL * m.sqrt(alpha2 + ((1.0f - alpha2) * NdotV) * NdotV);
    return m.div((2.0f * NdotL) * NdotV, denomA + denomB);
}
// :55-61
template <class M = Ieee>
__device__ __forceinline__ float G1_SmithGGX(float NdotV, float alpha, M m = M()) {
    float alpha2 = alpha * alpha;
    float denomC = m.sqrt(alpha2 + ((1.0f - alpha2) * NdotV) * NdotV) + NdotV;
    return m.div(2.0f * NdotV, denomC);
}
// :65-76
template <class M = Ieee>
__device__ __forceinline__ void CoordinateSystem(f3 N, f3& T, f3& B, M m = M()) {
    if (fabsf(N.z) < 0.999f) T = normalize3(cross3(mk3(0, 0, 1), N), m);
    else T = normalize3(cross3(mk3(1, 0, 0), N), m);
    B = cross3(N, T);
}
// :93-169
template <class M = Ieee>
__device__ __forceinline__ f3 SampleBRDF_GGX(const MatOpt& mat, f3 outgoing, f3 normal, uint2& seed, M m = M()) {
    float alpha = hmul(mat.Pr, mat.Pr);
    f3 N = normalize3(normal, m), V = normalize3(outgoing, m), T1, T2;
    CoordinateSystem(N, T1, T2, m);
    float vx = dot3(T1, V), vy = dot3(T2, V), vz = dot3(N, V);
    f3 Ve = normalize3(mk3(alpha * vx, alpha * vy, vz), m);
    float lensq = Ve.x * Ve.x + Ve.y * Ve.y;
    f3 T1h = (lensq > 0.0f) ? mk3(-Ve.y, Ve.x, 0.0f) * m.rsqrt(lensq) : mk3(1, 0, 0);
    f3 T2h = cross3(Ve, T1h);
    float U1 = RandomFloat(seed), U2 = RandomFloat(seed);
    float r = m.sqrt(U1);
    float phi = (2.0f * RTX_PI_REF) * U2;
    float sn, cs; d_sincos(phi, &sn, &cs);
    float t1 = r * cs, t2 = r * sn;
    float s = 0.5f * (1.0f + Ve.z);
    t2 = (1.0f - s) * m.sqrt(saturate1(1.0f - t1 * t1)) + s * t2;
    f3 Nh = (t1 * T1h + t2 * T2h) + m.sqrt(saturate1((1.0f - t1 * t1) - t2 * t2)) * Ve;
    f3 Ne = normalize3(mk3(alpha * Nh.x, alpha * Nh.y, fmaxf(0.0f, Nh.z)), m);
    f3 H = (Ne.x * T1 + Ne.y * T2) + Ne.z * N;
    f3 sample = reflect3(-V, H);
    if (dot3(sample, normal) < 0.0f) sample = -sample;
    return sample;
}
// :174-206
template <class M = Ieee>
__device__ __forceinline__ f3 EvaluateBRDF_GGX(const SceneData& S, const MatOpt& mat, f3 normal, f3 incoming, f3 outgoing, M m = M()) {
    f3 N = normalize3(normal, m), V = normalize3(outgoing, m), L = normalize3(-incoming, m);
    f3 H = normalize3(V + L, m);
    float NdotV = dot3(N, V), NdotL = dot3(N, L), NdotH = dot3(N, H), VdotH = dot3(V, H);
    f3 F = SchlickFresnel(mat.Ks, VdotH);
    float D = D_GGX(NdotH, mat.Pr, m);
    float G = G2_SmithGGX(NdotV, NdotL, hmul(mat.Pr, mat.Pr), m);
    float denominator = (4.0f * NdotV) * NdotL;
    if (denominator < RTX_EPS) return mk3(0, 0, 0);
    f3 specular = m.div3((F * D) * G, denominator);
    float Ess = ESS_LUT(S, mat, NdotV);
    float kms = m.div(1.0f - Ess, Ess);
    f3 specular_ess = specular * mk3(1.0f + mat.Ks.x * kms, 1.0f + mat.Ks.y * kms, 1.0f + mat.Ks.z * kms);
    if (any_nan_inf(specular_ess)) return mk3(0, 0, 0);
    return specular_ess;
}
// :209-224
template <class M = Ieee>
__device__ __forceinline__ float BRDF_PDF_GGX(const MatOpt& mat, f3 normal, f3 incoming, f3 outgoing, M m = M()) {
    f3 N = normalize3(normal, m), V = normalize3(outgoing, m), L = normalize3(-incoming, m);
    f3 H = normalize3(V + L, m);
    float NdotH = dot3(N, H), NdotV = dot3(N, V);
    float alpha = hmul(mat.Pr, mat.Pr);
    float G1 = G1_SmithGGX(NdotV, alpha, m);
    float D = D_GGX(NdotH, mat.Pr, m);
    return m.div(G1 * D, NdotV * 4.0f);
}

// ---- include/Lambertian_v6.hlsl
// :2-37
template <class M = Ieee>
__device__ __forceinline__ f3 RandomUnitVectorInHemisphere(f3 normal, uint2& seed, M m = M()) {
    float u1 = RandomFloat(seed), u2 = RandomFloat(seed);
    float r = m.sqrt(u1);
    float theta = (2.0f * 3.14159265358979323846f) * u2;
    float sn, cs; d_sincos(theta, &sn, &cs);
    float x = r * cs, y = r * sn;
    float z = m.sqrt(fmaxf(0.0f, (1.0f - x * x) - y * y));
    f3 h = normal;
    f3 up = fabsf(normal.z) < 0.999f ? mk3(0, 0, 1) : mk3(1, 0, 0);
    f3 right = normalize3(cross3(up, h), m);
    f3 forward = cross3(h, right);
    f3 hs = (x * right + y * forward) + z * h;
    hs = normalize3(hs, m);
    if (dot3(hs, normal) < 0.0f) hs = -hs;
    return hs;
}
// :51-58, :61-64
template <class M = Ieee>
__device__ __forceinline__ f3 EvaluateBRDF_Lambertian(const MatOpt& mat, M m = M()) { return m.div3k(mat.Kd, RTX_PI_REF, RTX_RCP_PI_REF); }
template <class M = Ieee>
__device__ __forceinline__ float BRDF_PDF_Lambertian(f3 normal, f3 incoming, M m = M()) {
    return m.divk(fmaxf(dot3(normal, -incoming), RTX_EPS), RTX_PI_REF, RTX_RCP_PI_REF);
}

// ---- shaders/BRDF_v7.hlsl
// :50-70
template <class M = Ieee>
__device__ __forceinline__ void CalculateStrategyProbabilities(const SceneData& S, const MatOpt& mat, f3 outgoing, f3 normal, float& p_d, float& p_s,
                                                               M m = M()) {
    if (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) { p_d = 1.0f; p_s = 0.0f; return; }
    float cosTheta = dot3(normal, outgoing);
    f3 fr = SchlickFresnel(mat.Ks, cosTheta);
    p_s = fminf(1.0f, m.divk((fr.x + fr.y) + fr.z, 3.0f, RTX_RCP_3) + mat.Pm);
    p_d = 1.0f - p_s;
}
// :7-48 (always one RandomFloat)
template <class M = Ieee>
__device__ __forceinline__ uint32_t SelectSamplingStrategy(const SceneData& S, const MatOpt& mat, f3 outgoing, f3 normal, uint2& seed, M m = M()) {
    float r = RandomFloat(seed);
    if (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) return 0;
    float cosTheta = dot3(normal, outgoing);
    f3 fr = SchlickFresnel(mat.Ks, cosTheta);
    float p_s = fminf(1.0f, m.divk((fr.x + fr.y) + fr.z, 3.0f, RTX_RCP_3) + mat.Pm);
    if (r <= p_s) { if (mat.Pr < 0.04f) return 0; return 1; }
    return 0;
}
// the two halves of SelectSamplingStrategy, for call sites that select twice at the same shading point
// (Path_Sampler_v7.hlsl:118,196): p_s depends on (material, outgoing, normal) only.
template <class M = Ieee>
__device__ __forceinline__ float StrategyPs(const SceneData& S, const MatOpt& mat, f3 outgoing, f3 normal, M m = M()) {
    if (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) return -1.0f;          // r <= p_s never holds: always strategy 0
    float cosTheta = dot3(normal, outgoing);
    f3 fr = SchlickFresnel(mat.Ks, cosTheta);
    return fminf(1.0f, m.divk((fr.x + fr.y) + fr.z, 3.0f, RTX_RCP_3) + mat.Pm);
}
__device__ __forceinline__ uint32_t SelectWithPs(float p_s, const MatOpt& mat, uint2& seed) {
    float r = RandomFloat(seed);
    if (r <= p_s) { if (mat.Pr < 0.04f) return 0; return 1; }
    return 0;
}
// :74-88
template <class M = Ieee>
__device__ __forceinline__ f3 SampleBRDF(uint32_t strategy, const MatOpt& mat, f3 outgoing, f3 normal, uint2& seed, M m = M()) {
    if (strategy == 0) return RandomUnitVectorInHemisphere(normal, seed, m);
    return SampleBRDF_GGX(mat, outgoing, normal, seed, m);
}
// the combined lobe F = p_d*f0 + p_s*f1 (Sampler_v7.hlsl:123-128,248-261,361-374,443-456,601-614; Path_Sampler_v7.hlsl:66-78)
template <class M = Ieee>
__device__ __forceinline__ f3 CombinedF(const SceneData& S, const MatOpt& mat, f3 normal, f3 incidence, f3 outgoing, float p_d, float p_s, M m = M()) {
    f3 F1 = SafeMultiply(p_d, EvaluateBRDF_Lambertian(mat, m));
    f3 F2 = (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) ? mk3(0, 0, 0) : SafeMultiply(p_s, EvaluateBRDF_GGX(S, mat, normal, incidence, outgoing, m));
    return F1 + F2;
}
// combined pdf with a common scale applied to each lobe before SafeMultiply: P = SM(p_d, pdf0*a/b) + SM(p_s, pdf1*a/b)
__device__ __forceinline__ float CombinedP_scaled(const SceneData& S, const MatOpt& mat, f3 normal, f3 incidence, f3 outgoing, float p_d,
                                                  float p_s, float a, float b) {
    float P1 = SafeMultiply1(p_d, (BRDF_PDF_Lambertian(normal, incidence) * a) / b);
    float P2 = (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) ? 0.0f : SafeMultiply1(p_s, (BRDF_PDF_GGX(mat, normal, incidence, outgoing) * a) / b);
    return P1 + P2;
}
__device__ __forceinline__ float CombinedP(const SceneData& S, const MatOpt& mat, f3 normal, f3 incidence, f3 outgoing, float p_d, float p_s) {
    float P1 = SafeMultiply1(p_d, BRDF_PDF_Lambertian(normal, incidence));
    float P2 = (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) ? 0.0f : SafeMultiply1(p_s, BRDF_PDF_GGX(mat, normal, incidence, outgoing));
    return P1 + P2;
}

// ---- the combined lobe with its shading-point invariants hoisted.
// CombinedF / CombinedP above are evaluated 5 times per path vertex (4 NEE candidates + the BSDF ray) with the same
// (material, normal, outgoing): N, V, N.V, the Smith term of V, G1, the D_GGX constants, the ESS energy factor and the
// Lambert lobe do not depend on the light direction.  LobeCtx computes them once; lobe_FP() then evaluates exactly the
// expression trees of EvaluateBRDF_GGX / BRDF_PDF_GGX / the Lambert lobe on those values (same operations on the same
// operands => bit-identical to the un-hoisted form, which tests/test_gpu_parity.py checks against the oracle).
struct LobeCtx {
    f3 normal;              // raw shading normal (the Lambert pdf uses it un-normalised)
    f3 N, V;                // normalize3(normal), normalize3(outgoing)
    f3 Ks, essScale;        // mat.Ks ; 1 + Ks*kms, kms = (1-Ess)/Ess (GGX_v7.hlsl:196-199)
    f3 F1;                  // SafeMultiply(p_d, Kd/PI)
    float NdotV, NdotV4;    // N.V ; 4*N.V
    float a2D, a2Dm1;       // D_GGX: alpha^2 with alpha = Pr*Pr in fp32 ; alpha^2 - 1
    float a2G, oma2G;       // Smith: alpha^2 with alpha = half(Pr*Pr) ; 1 - alpha^2
    float sV, G1;           // sqrt(a2G + ((1-a2G) N.V) N.V) ; (2 N.V)/(sV + N.V)
    float p_d, p_s;
    bool lambert_only;
};
// N = normalize3(normal) and V = normalize3(outgoing) supplied by the caller (call sites that build two contexts at one
// vertex share N, and often already hold V)
template <class M = Ieee>
__device__ __forceinline__ LobeCtx make_lobe_ctx_nv(const SceneData& S, const MatOpt& mat, f3 normal, f3 N, f3 V, float p_d, float p_s, M m = M()) {
    LobeCtx c;
    c.normal = normal; c.p_d = p_d; c.p_s = p_s;
    c.lambert_only = (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) != 0u;
    c.F1 = SafeMultiply(p_d, EvaluateBRDF_Lambertian(mat, m));
    c.Ks = mat.Ks;
    if (!c.lambert_only) {
        c.N = N; c.V = V;
        c.NdotV = dot3(c.N, c.V);
        c.NdotV4 = 4.0f * c.NdotV;
        const float alphaD = mat.Pr * mat.Pr;
        c.a2D = alphaD * alphaD; c.a2Dm1 = c.a2D - 1.0f;
        const float alphaG = hmul(mat.Pr, mat.Pr);
        c.a2G = alphaG * alphaG; c.oma2G = 1.0f - c.a2G;
        c.sV = m.sqrt(c.a2G + (c.oma2G * c.NdotV) * c.NdotV);
        c.G1 = m.div(2.0f * c.NdotV, c.sV + c.NdotV);
        const float Ess = ESS_LUT(S, mat, c.NdotV);
        const float kms = m.div(1.0f - Ess, Ess);
        c.essScale = mk3(1.0f + mat.Ks.x * kms, 1.0f + mat.Ks.y * kms, 1.0f + mat.Ks.z * kms);
    }
    return c;
}
template <class M = Ieee>
__device__ __forceinline__ LobeCtx make_lobe_ctx(const SceneData& S, const MatOpt& mat, f3 normal, f3 outgoing, float p_d, float p_s, M m = M()) {
    const bool lo = (S.cfg_flags & RTX_FLAG_LAMBERT_ONLY) != 0u;
    return make_lobe_ctx_nv(S, mat, normal, lo ? normal : normalize3(normal, m), lo ? outgoing : normalize3(outgoing, m), p_d, p_s, m);
}
// F = CombinedF(...), P = CombinedP(...) (scaled == false) or CombinedP_scaled(..., a, b) for one incidence direction.
template <bool WANT_F, bool WANT_P, class M = Ieee>
__device__ __forceinline__ void lobe_FP(const LobeCtx& c, f3 incidence, bool scaled, float a, float b, f3& F, float& P, M m = M()) {
    f3 F2 = mk3(0, 0, 0); float P2 = 0.0f;
    if (!c.lambert_only) {
        const f3 L = normalize3(-incidence, m);
        const f3 H = normalize3(c.V + L, m);
        const float NdotH = dot3(c.N, H);
        const float denomD = (NdotH * NdotH) * c.a2Dm1 + 1.0f;
        const float D = m.div(c.a2D, (RTX_PI_REF * denomD) * denomD);           // D_GGX
        if (WANT_F) {
            const float NdotL = dot3(c.N, L), VdotH = dot3(c.V, H);
            const f3 Fr = SchlickFresnel(c.Ks, VdotH);
            const float denomA = c.NdotV * m.sqrt(c.a2G + (c.oma2G * NdotL) * NdotL);
            const float denomB = NdotL * c.sV;
            const float G = m.div((2.0f * NdotL) * c.NdotV, denomA + denomB);   // G2_SmithGGX
            const float denominator = c.NdotV4 * NdotL;
            f3 spec = mk3(0, 0, 0);
            if (!(denominator < RTX_EPS)) {
                spec = m.div3((Fr * D) * G, denominator) * c.essScale;
                if (any_nan_inf(spec)) spec = mk3(0, 0, 0);
            }
            F2 = SafeMultiply(c.p_s, spec);
        }
        if (WANT_P) {
            float pdf = m.div(c.G1 * D, c.NdotV4);                                // BRDF_PDF_GGX (NdotV*4 == 4*NdotV)
            if (scaled) pdf = m.div(pdf * a, b);
            P2 = SafeMultiply1(c.p_s, pdf);
        }
    }
    if (WANT_F) F = c.F1 + F2;
    if (WANT_P) {
        float pl = BRDF_PDF_Lambertian(c.normal, incidence, m);
        if (scaled) pl = m.div(pl * a, b);
        P = SafeMultiply1(c.p_d, pl) + P2;
    }
}

// ---- ClosestHit, shaders/Hit_v7.hlsl:12-61 (area is not carried: nothing on the E0 path reads payload.area)
template <class MP = Ieee>
__device__ __forceinline__ void ClosestHit(const SceneData& S, f3 ro, f3 rd, float t, float b1, float b2, uint32_t prim, uint32_t inst, HitInfo& p,
                                           MP m = MP()) {
    const ModelRef M = S.models[S.inst_model[inst]];
    p.objID = inst;
    f3 worldOrigin = ro + t * rd;
    uint32_t vertId = 3u * prim;
    uint32_t mslot = vertId + M.mat_offset;
    uint32_t materialID = mslot < S.n_material_ids ? __ldg(&S.material_ids[mslot]) : 0u;
    float bary[3] = {(1.0f - b1) - b2, b1, b2};
    f3 pos[3], nrm[3];
    {
        const float4* r = M.shade + (size_t)prim * 5;
        // one record per hit out of 84 MB (C2): evict-first, like the path state (wave_dev.cuh StateView::ld)
        const float4 r0 = __ldcs(r), r1 = __ldcs(r + 1), r2 = __ldcs(r + 2), r3 = __ldcs(r + 3), r4 = __ldcs(r + 4);
        pos[0] = mk3(r0.x, r0.y, r0.z); pos[1] = mk3(r1.x, r1.y, r1.z); pos[2] = mk3(r2.x, r2.y, r2.z);
        nrm[0] = mk3(r0.w, r1.w, r2.w); nrm[1] = mk3(r3.x, r3.y, r3.z); nrm[2] = mk3(r4.x, r4.y, r4.z);
    }
    f3 e1 = pos[1] - pos[0], e2 = pos[2] - pos[0];
    f3 cross_a = cross3(e1, e2);
    f3 flatNormal = normalize3(cross_a, m);
    f3 smooth = mk3(0, 0, 0);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        if (nrm[i].x != 0.0f && nrm[i].y != 0.0f && nrm[i].z != 0.0f) smooth = smooth + nrm[i] * bary[i];
        else smooth = smooth + flatNormal * bary[i];
    }
    f3 normal;
    if (length3(smooth, m) > 0.0001f) normal = normalize3(smooth, m); else normal = flatNormal;
    f3 wn = mul43(S.props[inst].objectToWorldNormal, normal.x, normal.y, normal.z, 0.0f);
    p.hitNormal = normalize3(wn, m);
    p.materialID = materialID;
    p.hitPosition = worldOrigin;
}

// ---- shaders/Sampler_v7.hlsl
// :106-131
template <class M = Ieee>
__device__ __forceinline__ f3 ReconnectDI(const SceneData& S, f3 x1, f3 n1, f3 x2, f3 n2, f3 L, f3 outgoing, const MatOpt& material, M m = M()) {
    f3 dir = x2 - x1;
    float dist = length3(dir, m);
    float cosThetaX1 = fmaxf(0.0f, dot3(n1, normalize3(dir, m)));
    if (dot3(n2, normalize3(-dir, m)) < 0.0f) n2 = -n2;
    float cosThetaX2 = fmaxf(0.0f, dot3(n2, normalize3(-dir, m)));
    float p_d, p_s;
    CalculateStrategyProbabilities(S, material, normalize3(outgoing, m), n1, p_d, p_s, m);
    f3 F = CombinedF(S, material, n1, normalize3(-dir, m), normalize3(outgoing, m), p_d, p_s, m);
    return m.div3(((F * L) * cosThetaX1) * cosThetaX2, dist * dist);
}
// :134-161
template <class M = Ieee>
__device__ __forceinline__ f3 ReconnectGI(const SceneData& S, f3 x1, f3 n1, f3 x2, f3 L, f3 outgoing, const MatOpt& material1, M m = M()) {
    f3 dir = x2 - x1;
    float cosThetaX1 = fabsf(dot3(n1, normalize3(dir, m)));
    float p_d, p_s;
    CalculateStrategyProbabilities(S, material1, normalize3(outgoing, m), n1, p_d, p_s, m);
    f3 Fx1 = CombinedF(S, material1, n1, normalize3(-dir, m), normalize3(outgoing, m), p_d, p_s, m);
    f3 fr = (Fx1 * cosThetaX1) * L;
    if (any_nan_inf(fr)) return mk3(0, 0, 0);
    return fr;
}

// light selection :293-308
__device__ __forceinline__ uint32_t SelectLight(const SceneData& S, float randomValue) {
    int left = 0, right = (int)__ldg(&S.lights[0].triCount) - 1, selected = 0;
    while (left <= right) {
        int mid = left + (right - left) / 2;
        if (randomValue < __ldg(&S.lights[mid].cdf)) { selected = mid; right = mid - 1; }
        else left = mid + 1;
    }
    return (uint32_t)selected;
}

struct LightSample { f3 point, normal_l, L_norm, emission; float dist2, pdf_l; };

// shared front half of SampleLightNEE (:292-346) and SampleLightNEE_GI (:529-584): 3 RandomFloat
template <class MP = Ieee>
__device__ __forceinline__ void SampleLightPoint(const SceneData& S, f3 origin, uint2& seed, LightSample& ls, MP m = MP()) {
    float randomValue = RandomFloat(seed);
    const float4* lt = reinterpret_cast<const float4*>(S.lights + SelectLight(S, randomValue));
    const float4 l0 = __ldg(lt), l1 = __ldg(lt + 1), l2 = __ldg(lt + 2), l3 = __ldg(lt + 3);
    const float* M = S.props[__float_as_uint(l1.w)].objectToWorld;
    f3 x_v = mul43(M, l0.x, l0.y, l0.z, 1.0f);
    f3 y_v = mul43(M, l1.x, l1.y, l1.z, 1.0f);
    f3 z_v = mul43(M, l2.x, l2.y, l2.z, 1.0f);
    float xi1 = RandomFloat(seed), xi2 = RandomFloat(seed);
    if (xi1 + xi2 > 1.0f) { xi1 = 1.0f - xi1; xi2 = 1.0f - xi2; }
    float u = (1.0f - xi1) - xi2, v = xi1, w = xi2;
    ls.point = (u * x_v + v * y_v) + w * z_v;
    f3 L = ls.point - origin;
    ls.dist2 = dot3(L, L);
    ls.L_norm = normalize3(L, m);
    f3 cross_l = cross3(y_v - x_v, z_v - x_v);
    f3 normal_l = normalize3(cross_l, m);
    if (dot3(normal_l, -ls.L_norm) < 0.0f) normal_l = -normal_l;
    ls.normal_l = normal_l;
    float area_l = fabsf(length3(cross_l, m) * 0.5f);
    ls.pdf_l = m.div(l2.w, fmaxf(area_l, RTX_EPS));
    ls.emission = mk3(l3.x, l3.y, l3.z);
}

}  // namespace rtx
