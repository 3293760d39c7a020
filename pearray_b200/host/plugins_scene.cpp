// Entity, camera, emission, infinite-light, sampler, filter, spectral-mapper and integrator plugins of the
// hot path (SURVEY rows 13,16-20,22,23).  Names, aliases, parameter keys and defaults follow the reference.
#include "prh.h"

#include <sstream>

namespace PR {
namespace {
// ------------------------------------------------------------------ entities
class MeshEntity : public IEntity { // plugins/main/entities/mesh.cpp:130-256
public:
	MeshEntity(const std::string& name, const Transformf& t, const std::shared_ptr<MeshBase>& mesh, const std::vector<uint32>& materials, uint32 emsID)
		: IEntity(emsID, name, t)
		, mMaterials(materials)
		, mMesh(mesh)
	{
	}
	std::string type() const override { return "mesh"; }
	float localSurfaceArea() const override { return mMesh->surfaceArea(Transformf::Identity()); }
	BoundingBox worldBoundingBox() const override
	{
		BoundingBox b;
		for (size_t i = 0; i < mMesh->vertexCount(); ++i)
			b.combine(transform() * mMesh->vertex((uint32)i));
		return b;
	}
	void describe(prb_entity& out, SceneCompiler& c) const override
	{
		out.type			= PRB_ENTITY_MESH;
		out.mesh_id			= c.registerMesh(mMesh);
		out.material_offset = c.registerEntityMaterials(mMaterials);
		out.material_count	= (uint32)mMaterials.size();
	}

private:
	std::vector<uint32> mMaterials;
	std::shared_ptr<MeshBase> mMesh;
};
class MeshEntityPlugin : public IEntityPlugin {
public:
	std::shared_ptr<IEntity> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		const std::string name		 = params.getString("name", "__unnamed__");
		const std::string mesh_name	 = params.getString("mesh", "");
		Parameter matP				 = params.getParameter("materials");
		if (!matP.isValid())
			matP = params.getParameter("material");
		const std::vector<uint32> materials = ctx.lookupMaterialIDArray(matP);
		const uint32 emsID					= ctx.lookupEmissionID(params.getParameter("emission"));
		if (params.getBool("ignore_normals", false))
			PR_LOG(L_WARNING) << "mesh: ignore_normals is not supported on the device path (vertex normals are used when present)" << std::endl;
		if (!ctx.hasMesh(mesh_name)) {
			PR_LOG(L_ERROR) << "Could not find a mesh named " << mesh_name << std::endl;
			return nullptr;
		}
		return std::make_shared<MeshEntity>(name, ctx.transform(), ctx.getMesh(mesh_name), materials, emsID);
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "mesh" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Mesh Entity: mesh, material|materials, emission, ignore_normals"; }
};

class SphereEntity : public IEntity { // sphere.cpp:19-153
public:
	SphereEntity(const std::string& name, const Transformf& t, float r, uint32 matID, uint32 emsID)
		: IEntity(emsID, name, t)
		, mRadius(r)
		, mMaterialID(matID)
	{
		mPDF_Cache = r > PR_EPSILON ? 1 / worldSurfaceArea() : 0.0f;
	}
	std::string type() const override { return "sphere"; }
	float localSurfaceArea() const override { return 4 * PR_PI * mRadius * mRadius; }
	float worldSurfaceArea() const override
	{ // Knud Thomsen's formula, sphere.cpp:47-61
		constexpr float P = 1.6075f;
		const Vector3f s  = transform().scaling();
		const float a = s.x * mRadius, b = s.y * mRadius, c = s.z * mRadius;
		const float t = (std::pow(a * b, P) + std::pow(a * c, P) + std::pow(b * c, P)) / 3;
		return 4 * PR_PI * std::pow(t, 1 / P);
	}
	float worldRadius() const
	{
		const Matrix3f& L = transform().linear();
		return mRadius * ((L.col(0).norm() + L.col(1).norm() + L.col(2).norm()) / 3.0f);
	}
	BoundingBox worldBoundingBox() const override
	{
		const Vector3f c = transform() * Vector3f(0, 0, 0);
		const float r	 = worldRadius();
		BoundingBox b;
		b.combine(c - Vector3f(r, r, r));
		b.combine(c + Vector3f(r, r, r));
		return b;
	}
	float sampleParameterPointPDF() const override { return mPDF_Cache; }
	void describe(prb_entity& out, SceneCompiler& c) const override
	{
		out.type			= PRB_ENTITY_SPHERE;
		out.material_offset = c.registerEntityMaterials({ mMaterialID });
		out.material_count	= 1;
		const Vector3f ctr	= transform() * Vector3f(0, 0, 0);
		out.geo[0]			= ctr.x;
		out.geo[1]			= ctr.y;
		out.geo[2]			= ctr.z;
		out.geo[3]			= worldRadius();
		out.geo[4]			= mRadius;
		out.geo[5]			= mPDF_Cache;
	}

private:
	float mRadius;
	uint32 mMaterialID;
	float mPDF_Cache;
};
class SphereEntityPlugin : public IEntityPlugin {
public:
	std::shared_ptr<IEntity> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		return std::make_shared<SphereEntity>(params.getString("name", "__unnamed__"), ctx.transform(), params.getNumber("radius", 1.0f),
											  ctx.lookupMaterialID(params.getParameter("material")), ctx.lookupEmissionID(params.getParameter("emission")));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "sphere" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Sphere Entity: radius (1), material, emission, optimize_sampling (true)"; }
};

class PlaneEntity : public IEntity { // plane.cpp:18-258
public:
	PlaneEntity(const std::string& name, const Transformf& t, const Vector3f& xAxis, const Vector3f& yAxis, uint32 matID, uint32 emsID, bool centering)
		: IEntity(emsID, name, t)
		, mPos(0, 0, 0)
		, mX(xAxis)
		, mY(yAxis)
		, mMaterialID(matID)
	{
		if (centering)
			mPos = -0.5f * mX - 0.5f * mY;
	}
	Vector3f normal() const { return mX.cross(mY).normalized(); }
	std::string type() const override { return "plane"; }
	float localSurfaceArea() const override { return mX.cross(mY).norm(); }
	float worldSurfaceArea() const override { return (transform().linear() * mX).norm() * (transform().linear() * mY).norm(); }
	BoundingBox worldBoundingBox() const override
	{
		BoundingBox b;
		b.combine(transform() * mPos);
		b.combine(transform() * (mPos + mY));
		b.combine(transform() * (mPos + mY + mX));
		b.combine(transform() * (mPos + mX));
		return b;
	}
	float sampleParameterPointPDF() const override
	{
		const float garea = worldSurfaceArea();
		return garea > PR_EPSILON ? 1.0f / garea : 0;
	}
	void describe(prb_entity& out, SceneCompiler& c) const override
	{
		out.type			= PRB_ENTITY_PLANE;
		out.material_offset = c.registerEntityMaterials({ mMaterialID });
		out.material_count	= 1;
		// cache(), plane.cpp:227-244
		const Vector3f S = transform() * mPos;
		Vector3f Ex = transform().linear() * mX, Ey = transform().linear() * mY, Ez = normalMatrix() * normal();
		const float w = Ex.norm(), h = Ey.norm();
		Ex.normalize();
		Ey.normalize();
		Ez.normalize();
		auto put = [&](int o, const Vector3f& v) {
			out.geo[o]	   = v.x;
			out.geo[o + 1] = v.y;
			out.geo[o + 2] = v.z;
		};
		put(0, S);
		put(3, Ex);
		put(6, Ey);
		put(9, Ez);
		out.geo[12] = w;
		out.geo[13] = h;
		put(14, transform() * mPos); // constructGeometryRepresentation, plane.cpp:80-84
		put(17, transform() * (mPos + mY));
		put(20, transform() * (mPos + mY + mX));
		put(23, transform() * (mPos + mX));
		put(26, normalMatrix() * normal());
		put(29, mPos);
		put(32, mX);
		put(35, mY);
		out.geo[38] = 1 / mX.squaredNorm();
		out.geo[39] = 1 / mY.squaredNorm();
	}

private:
	Vector3f mPos, mX, mY;
	uint32 mMaterialID;
};
class PlaneEntityPlugin : public IEntityPlugin {
public:
	std::shared_ptr<IEntity> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		Vector3f xAxis				 = params.getVector3f("x_axis", Vector3f(1, 0, 0));
		Vector3f yAxis				 = params.getVector3f("y_axis", Vector3f(0, 1, 0));
		const float width			 = params.getNumber("width", 1);
		const float height			 = params.getNumber("height", 1);
		return std::make_shared<PlaneEntity>(params.getString("name", "__unnamed__"), ctx.transform(), width * xAxis, height * yAxis,
											 ctx.lookupMaterialID(params.getParameter("material")), ctx.lookupEmissionID(params.getParameter("emission")),
											 params.getBool("centering", false));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "plane" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Plane Entity: width (1), height (1), x_axis, y_axis, material, emission, centering (false)"; }
};

// ------------------------------------------------------------------ camera
class PerspectiveCamera : public ICamera { // plugins/main/cameras/perspective.cpp:15-137 (both the HasDOF and the pinhole form)
public:
	PerspectiveCamera(const std::string& name, const Transformf& t, float w, float h, float fstop, float apert, float nearT, float farT, const Vector3f& ld,
					  const Vector3f& lr, const Vector3f& lu)
		: ICamera(name, t)
		, mWidth(w)
		, mHeight(h)
		, mFStop(fstop)
		, mApertureRadius(apert)
		, mNearT(nearT)
		, mFarT(farT)
		, mLD(ld)
		, mLR(lr)
		, mLU(lu)
	{
	}
	std::string type() const override { return "perspective"; }
	void describe(prb_camera& out) const override
	{ // cache(), perspective.cpp:84-113
		const bool hasDOF = mApertureRadius > PR_EPSILON && mFStop > PR_EPSILON; // PerspectiveCameraPlugin::create, :156
		Vector3f dir	  = transform().linear() * mLD;
		Vector3f right	  = transform().linear() * mLR;
		Vector3f up		  = transform().linear() * mLU;
		Vector3f apx(0, 0, 0), apy(0, 0, 0);
		if (!hasDOF) {
			right = right * (0.5f * mWidth);
			up	  = up * (0.5f * mHeight);
		} else {
			dir	  = dir * (mFStop + 1); // mFocalDistance_Cache
			apx	  = right * mApertureRadius;
			apy	  = up * mApertureRadius;
			right = right * (0.5f * mWidth * (mFStop + 1));
			up	  = up * (0.5f * mHeight * (mFStop + 1));
		}
		const Vector3f o = transform().translation();
		for (int i = 0; i < 3; ++i) {
			out.origin[i]	  = o[i];
			out.right[i]	  = right[i];
			out.up[i]		  = up[i];
			out.dir[i]		  = dir[i];
			out.aperture_x[i] = apx[i];
			out.aperture_y[i] = apy[i];
		}
		out.near_t	= mNearT;
		out.far_t	= mFarT;
		out.type	= PRB_CAMERA_PERSPECTIVE;
		out.has_dof = hasDOF ? 1u : 0u;
	}

private:
	float mWidth, mHeight, mFStop, mApertureRadius, mNearT, mFarT;
	Vector3f mLD, mLR, mLU;
};
class OrthoCamera : public ICamera { // plugins/main/cameras/ortho.cpp:15-84
public:
	OrthoCamera(const std::string& name, const Transformf& t, float w, float h, float nearT, float farT, const Vector3f& ld, const Vector3f& lr, const Vector3f& lu)
		: ICamera(name, t)
		, mWidth(w)
		, mHeight(h)
		, mNearT(nearT)
		, mFarT(farT)
		, mLD(ld)
		, mLR(lr)
		, mLU(lu)
	{
	}
	std::string type() const override { return "orthographic"; }
	void describe(prb_camera& out) const override
	{ // the cached members of the constructor, ortho.cpp:29-31: the direction is normalised, right / up carry half the extent
		const Vector3f dir	 = (transform().linear() * mLD).normalized();
		const Vector3f right = (transform().linear() * mLR) * 0.5f * mWidth;
		const Vector3f up	 = (transform().linear() * mLU) * 0.5f * mHeight;
		const Vector3f o	 = transform().translation();
		for (int i = 0; i < 3; ++i) {
			out.origin[i] = o[i];
			out.right[i]  = right[i];
			out.up[i]	  = up[i];
			out.dir[i]	  = dir[i];
		}
		out.near_t = mNearT;
		out.far_t  = mFarT;
		out.type   = PRB_CAMERA_ORTHOGRAPHIC;
	}

private:
	float mWidth, mHeight, mNearT, mFarT;
	Vector3f mLD, mLR, mLU;
};
class OrthoCameraPlugin : public ICameraPlugin {
public:
	std::shared_ptr<ICamera> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		return std::make_shared<OrthoCamera>(params.getString("name", "__unnamed__"), ctx.transform(), params.getNumber("width", 1), params.getNumber("height", 1),
											 params.getNumber("near", 0.000001f), params.getNumber("far", PR_INF),
											 params.getVector3f("local_direction", Vector3f(0, 1, 0)), params.getVector3f("local_right", Vector3f(1, 0, 0)),
											 params.getVector3f("local_up", Vector3f(0, 0, 1)));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "ortho", "orthographic" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Orthogonal Camera: width, height, near, far, local_direction, local_right, local_up"; }
};
class PerspectiveCameraPlugin : public ICameraPlugin {
public:
	std::shared_ptr<ICamera> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		const float apr				 = params.getNumber("aperture_radius", 0.05f);
		const float fstop			 = params.getNumber("fstop", 0);
		// ICamera::DefaultDirection (0,1,0) /Right (1,0,0) /Up (0,0,1) (src/core/camera/ICamera.cpp:5-7) and NEAR/FAR defaults (perspective.cpp:12-13)
		return std::make_shared<PerspectiveCamera>(params.getString("name", "__unnamed__"), ctx.transform(), params.getNumber("width", 1),
												   params.getNumber("height", 1), fstop, apr, params.getNumber("near", 0.000001f), params.getNumber("far", PR_INF),
												   params.getVector3f("local_direction", Vector3f(0, 1, 0)), params.getVector3f("local_right", Vector3f(1, 0, 0)),
												   params.getVector3f("local_up", Vector3f(0, 0, 1)));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "standard_camera", "standard", "default", "perspective" });
		return names;
	}
	std::string specification(const std::string&) const override
	{
		return "Perspective Camera: width, height, fstop (0), aperture_radius (0.05), near, far, local_direction, local_right, local_up";
	}
};

// ------------------------------------------------------------------ emission
class DiffuseEmission : public IEmission { // plugins/main/emissions/diffuse.cpp:11-56
public:
	explicit DiffuseEmission(const std::shared_ptr<FloatSpectralNode>& spec)
		: mRadiance(spec)
	{
	}
	SpectralBlob power(const SpectralBlob& wvl) const override { return NodeUtils::average(wvl, mRadiance.get()); }
	SpectralRange spectralRange() const override { return mRadiance->spectralRange(); }
	void describe(prb_emission& out, NodeEmitter& e) const override { out.radiance_node = mRadiance->emit(e); }
	std::string dumpInformation() const override { return "  <DiffuseEmission>: " + mRadiance->dumpInformation() + "\n"; }

private:
	std::shared_ptr<FloatSpectralNode> mRadiance;
};
class DiffuseEmissionPlugin : public IEmissionPlugin {
public:
	std::shared_ptr<IEmission> create(const std::string&, const SceneLoadContext& ctx) override
	{
		return std::make_shared<DiffuseEmission>(ctx.lookupSpectralNode("radiance", 1));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "diffuse", "standard", "default" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Diffuse Emission: radiance (spectral, 1)"; }
};

// ------------------------------------------------------------------ environment light
class EnvironmentLight : public IInfiniteLight { // plugins/main/infinitelights/environment.cpp:24-146
public:
	EnvironmentLight(const std::string& name, const Transformf& t, const std::shared_ptr<FloatSpectralNode>& rad, const std::shared_ptr<FloatSpectralNode>& bg,
					 bool allowDistribution)
		: IInfiniteLight(name, t)
		, mRadiance(rad)
		, mBackground(bg)
	{
		// EnvironmentLightFactory::create, environment.cpp:172-198: an image based radiance gets a Distribution2D of its size
		int w = 1, h = 1;
		mRadiance->queryRecommendedSize(w, h);
		if (allowDistribution && w > 1 && h > 1) {
			mW = w;
			mH = h;
			std::vector<float> integrals(mH, 0.0f);
			mConditional.assign(mH, Distribution1D(mW));
			for (int y = 0; y < mH; ++y)
				mConditional[y].generate(
					[&](size_t x) {
						const float u		 = (x + 0.5f) / (float)mW;
						const float v		 = (y + 0.5f) / (float)mH;
						const float sinTheta = std::sin(PR_PI * v);
						ShadingContext coord;
						coord.UV		   = Vector2f(u, v);
						coord.WavelengthNM = SpectralBlob(560.0f, 540.0f, 400.0f, 600.0f); // preset of wavelengths to test
						const SpectralBlob r = mRadiance->eval(coord);
						const float val		 = sinTheta * std::max(std::max(r[0], r[1]), std::max(r[2], r[3]));
						return (val <= PR_EPSILON) ? 0.0f : val;
					},
					&integrals[y]);
			mMarginal = Distribution1D(mH);
			mMarginal.generate([&](size_t y) { return integrals[y]; });
		}
	}
	SpectralBlob power(const SpectralBlob& wvl) const override { return NodeUtils::average(wvl, mRadiance.get()); }
	SpectralRange spectralRange() const override { return mRadiance->spectralRange(); }
	void describe(prb_light& out, NodeEmitter& e) const override
	{
		out.type			= PRB_LIGHT_ENV;
		out.radiance_node	= mRadiance->emit(e);
		out.background_node = mBackground->emit(e);
		out.env_split		= mRadiance != mBackground;
		for (int i = 0; i < 9; ++i) {
			out.normal_matrix[i]	 = normalMatrix().m[i];
			out.inv_normal_matrix[i] = invNormalMatrix().m[i];
		}
		if (mW > 0) { // marginal CDF, then one conditional CDF per row (the layout of the sky light's Distribution2D)
			std::vector<float>& pool = *e.pool;
			out.dist_offset			 = (uint32)pool.size();
			out.dist_w				 = (uint32)mW;
			out.dist_h				 = (uint32)mH;
			pool.insert(pool.end(), mMarginal.cdf().begin(), mMarginal.cdf().end());
			for (int y = 0; y < mH; ++y)
				pool.insert(pool.end(), mConditional[y].cdf().begin(), mConditional[y].cdf().end());
		}
	}

private:
	std::shared_ptr<FloatSpectralNode> mRadiance, mBackground;
	int mW = 0, mH = 0;
	std::vector<Distribution1D> mConditional;
	Distribution1D mMarginal;
};
class EnvironmentLightFactory : public IInfiniteLightPlugin {
public:
	std::shared_ptr<IInfiniteLight> create(const std::string&, const SceneLoadContext& ctx) override
	{
		const ParameterGroup& params = ctx.parameters();
		const auto radP				 = params.getParameter("radiance");
		const auto backgroundP		 = params.getParameter("background");
		std::shared_ptr<FloatSpectralNode> radiance, background;
		if (radP.isValid() && backgroundP.isValid()) {
			radiance   = ctx.lookupSpectralNode(radP, 1);
			background = ctx.lookupSpectralNode(backgroundP, 1);
		} else if (radP.isValid()) {
			radiance   = ctx.lookupSpectralNode(radP, 1);
			background = radiance;
		} else {
			background = ctx.lookupSpectralNode(backgroundP, 1);
			radiance   = background;
		}
		if (params.getBool("compensation", false))
			throw std::runtime_error("env: ':compensation true' (MIS compensation, off by default in the reference) is not supported");
		return std::make_shared<EnvironmentLight>(params.getString("name", "__unknown"), ctx.transform(), radiance, background, params.getBool("distribution", true));
	}
	const std::vector<std::string>& getNames() const override
	{
		static std::vector<std::string> names({ "env", "environment", "background" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Environment Light: radiance (spectral, 1), background (spectral)"; }
};

// ------------------------------------------------------------------ samplers
constexpr uint32 DEF_SAMPLE_COUNT = 128;
class RandomSampler : public ISampler { // RandomSampler.cpp:11-22
public:
	using ISampler::ISampler;
	float generate1D(Random& rnd, uint32) override { return rnd.getFloat(); }
	Vector2f generate2D(Random& rnd, uint32) override { return rnd.get2D(); }
	void describe(prb_sampler& out, std::vector<float>&) const override
	{
		out.type		= PRB_SAMPLER_RANDOM;
		out.max_samples = maxSamples();
	}
};
inline uint32 mj_permute(uint32 i, uint32 l, uint32 p)
{ // Kensler, Correlated Multi-Jittered Sampling (MultiJitteredSampler.cpp:21-76)
	uint32 w = l - 1;
	if (w == 0)
		return 0;
	const bool pow2 = (l & w) == 0;
	if (!pow2) {
		w |= w >> 1;
		w |= w >> 2;
		w |= w >> 4;
		w |= w >> 8;
		w |= w >> 16;
	}
	do {
		i ^= p;
		i *= 0xe170893d;
		i ^= p >> 16;
		i ^= (i & w) >> 4;
		i ^= p >> 8;
		i *= 0x0929eb3f;
		i ^= p >> 23;
		i ^= (i & w) >> 1;
		i *= 1 | p >> 27;
		i *= 0x6935fa69;
		i ^= (i & w) >> 11;
		i *= 0x74dcb303;
		i ^= (i & w) >> 2;
		i *= 0x9e501cc3;
		i ^= (i & w) >> 2;
		i *= 0xc860a3df;
		i &= w;
		i ^= i >> 5;
	} while (!pow2 && i >= l);
	return pow2 ? ((i + p) & w) : ((i + p) % l);
}
class MultiJitteredSampler : public ISampler { // MultiJitteredSampler.cpp:95-157
public:
	MultiJitteredSampler(uint32 samples, uint32 bins, uint32 seed)
		: ISampler(samples)
		, m1D(bins)
		, m2D_X(static_cast<uint32>(std::sqrt(bins)))
		, m2D_Y((bins + m2D_X - 1) / m2D_X)
		, mSeed(seed)
	{
	}
	float generate1D(Random& rnd, uint32 index) override
	{
		const float j = rnd.getFloat();
		return (index % m1D + j) / m1D;
	}
	Vector2f generate2D(Random& rnd, uint32 index) override
	{
		constexpr uint32 FH = 0x51633e2d, F1 = 0x68bc21eb, F2 = 0x02e5be93;
		index			= mj_permute(index, std::max(1u, maxSamples()), mSeed * FH);
		const uint32 sx = mj_permute(index % m2D_X, m2D_X, mSeed * F1);
		const uint32 sy = mj_permute(index / m2D_X, m2D_Y, mSeed * F2);
		const float jx	= rnd.getFloat();
		const float jy	= rnd.getFloat();
		return Vector2f((sx + (sy + jx) / m2D_Y) / m2D_X, (index + jy) / std::max(1u, maxSamples()));
	}
	void describe(prb_sampler& out, std::vector<float>&) const override
	{
		out.type		= PRB_SAMPLER_MJITT;
		out.max_samples = maxSamples();
		out.bins_1d		= m1D;
		out.m2d_x		= m2D_X;
		out.m2d_y		= m2D_Y;
		out.seed		= mSeed;
	}

private:
	uint32 m1D, m2D_X, m2D_Y, mSeed;
};
class SobolSampler : public ISampler { // SobolSampler.cpp:27-78
public:
	SobolSampler(Random& random, uint32 samples)
		: ISampler(samples)
	{
		// direction numbers: dim 0 = van der Corput (2^(63-i)); dim 1 = Sobol' polynomial x+1, v_i = v_{i-1} ^ (v_{i-1} >> 1)
		// (identical to the first two rows of SobolSamplerData.inl)
		uint64 V0[64], V1[64];
		for (int i = 0; i < 64; ++i)
			V0[i] = 1ULL << (63 - i);
		V1[0] = 1ULL << 63;
		for (int i = 1; i < 64; ++i)
			V1[i] = V1[i - 1] ^ (V1[i - 1] >> 1);
		std::vector<float> s1(samples, 0.0f);
		std::vector<Vector2f> s2(samples);
		uint64 last[2] = { 0, 0 };
		for (uint32 i = 1; i < samples; ++i) {
			uint32 n	= i - 1;
			size_t cin	= 1; // index from the right of the first zero bit
			while (n & 1) {
				n >>= 1;
				++cin;
			}
			last[0] ^= V0[cin - 1];
			last[1] ^= V1[cin - 1];
			s1[i] = static_cast<float>(Random::uint64ToDouble(last[0]));
			s2[i] = Vector2f(s1[i], static_cast<float>(Random::uint64ToDouble(last[1])));
		}
		// std::shuffle(m1D, rnd); std::shuffle(m2D, rnd)  (libstdc++ semantics, prh core.cpp)
		std::vector<uint32> perm(samples);
		for (uint32 i = 0; i < samples; ++i)
			perm[i] = i;
		libstdcxxShuffle(perm, random);
		mSamples1D.resize(samples);
		for (uint32 i = 0; i < samples; ++i)
			mSamples1D[i] = s1[perm[i]];
		for (uint32 i = 0; i < samples; ++i)
			perm[i] = i;
		libstdcxxShuffle(perm, random);
		mSamples2D.resize(samples);
		for (uint32 i = 0; i < samples; ++i)
			mSamples2D[i] = s2[perm[i]];
	}
	float generate1D(Random& rnd, uint32 index) override { return mSamples1D.size() <= index ? rnd.getFloat() : mSamples1D[index]; }
	Vector2f generate2D(Random& rnd, uint32 index) override { return mSamples2D.size() <= index ? rnd.get2D() : mSamples2D[index]; }
	void describe(prb_sampler& out, std::vector<float>& pool) const override
	{
		out.type		 = PRB_SAMPLER_SOBOL;
		out.max_samples	 = maxSamples();
		out.table_offset = (uint32)pool.size();
		pool.insert(pool.end(), mSamples1D.begin(), mSamples1D.end());
		for (const auto& v : mSamples2D) {
			pool.push_back(v.x);
			pool.push_back(v.y);
		}
	}

private:
	std::vector<float> mSamples1D;
	std::vector<Vector2f> mSamples2D;
};
class StratifiedSampler : public ISampler { // StratifiedSampler.cpp:12-41, Projection::stratified (src/base/math/Projection.h:14-18)
public:
	StratifiedSampler(uint32 samples, uint32 groups)
		: ISampler(samples)
		, m2D_X(static_cast<uint32>(std::sqrt(groups)))
		, mGroups(groups)
	{
	}
	static float stratified(float u, int index, int groups)
	{
		const float range = 1.0f / groups;
		return u * range + index * range;
	}
	float generate1D(Random& rnd, uint32 index) override { return stratified(rnd.getFloat(), (int)index, (int)mGroups); }
	Vector2f generate2D(Random& rnd, uint32 index) override
	{
		const float x = stratified(rnd.getFloat(), (int)(index % m2D_X), (int)m2D_X);
		const float y = stratified(rnd.getFloat(), (int)(index / m2D_X), (int)m2D_X);
		return Vector2f(x, y);
	}
	void describe(prb_sampler& out, std::vector<float>&) const override
	{
		out.type		= PRB_SAMPLER_STRATIFIED;
		out.max_samples = maxSamples();
		out.bins_1d		= mGroups;
		out.m2d_x		= m2D_X;
	}

private:
	uint32 m2D_X, mGroups;
};
class UniformSampler : public ISampler { // UniformSampler.cpp:11-29 ("a very bad sampler for test purposes")
public:
	using ISampler::ISampler;
	float generate1D(Random&, uint32) override { return 0.5f; }
	Vector2f generate2D(Random&, uint32) override { return Vector2f(0.5f, 0.5f); }
	void describe(prb_sampler& out, std::vector<float>&) const override
	{
		out.type		= PRB_SAMPLER_UNIFORM;
		out.max_samples = maxSamples();
	}
};
inline float haltonValue(uint32 index, uint32 base)
{ // radical inverse as the reference computes it (fp32), HaltonSampler.cpp:14-25
	float result = 0;
	float f		 = 1;
	for (uint32 i = index; i > 0;) {
		f = f / base;
		result += f * (i % base);
		i = static_cast<uint32>(std::floor(i / static_cast<float>(base)));
	}
	return result;
}
class HaltonSampler : public ISampler { // HaltonSampler (:30-72) and HammersleySampler (:77-121): y = (0.5 + i) / samples inside the table
public:
	HaltonSampler(uint32 samples, uint32 baseX, uint32 baseY, uint32 burnin, bool hammersley)
		: ISampler(samples)
		, mX(samples)
		, mY(samples)
		, mBaseX(baseX)
		, mBaseY(hammersley ? 47u /* HAMMERSLEY_EVASIVE_BASE_Y */ : baseY)
		, mBurnin(burnin)
	{
		for (uint32 i = 0; i < samples; ++i) {
			mX[i] = haltonValue(i + burnin, baseX);
			mY[i] = hammersley ? (0.5f + i) / samples : haltonValue(i + burnin, baseY);
		}
	}
	float generate1D(Random&, uint32 index) override { return index < maxSamples() ? mX[index] : haltonValue(index + mBurnin, mBaseX); }
	Vector2f generate2D(Random&, uint32 index) override
	{
		if (index < maxSamples())
			return Vector2f(mX[index], mY[index]);
		return Vector2f(haltonValue(index + mBurnin, mBaseX), haltonValue(index + mBurnin, mBaseY));
	}
	void describe(prb_sampler& out, std::vector<float>& pool) const override
	{
		out.type		 = PRB_SAMPLER_HALTON;
		out.max_samples	 = maxSamples();
		out.m2d_x		 = mBaseX;
		out.m2d_y		 = mBaseY;
		out.seed		 = mBurnin;
		out.table_offset = (uint32)pool.size();
		pool.insert(pool.end(), mX.begin(), mX.end());
		for (uint32 i = 0; i < maxSamples(); ++i) {
			pool.push_back(mX[i]);
			pool.push_back(mY[i]);
		}
	}

private:
	std::vector<float> mX, mY;
	uint32 mBaseX, mBaseY, mBurnin;
};
enum class SamplerKind { Random, MJitt, Sobol, Stratified, Uniform, Halton, Hammersley };
class SamplerFactory : public ISamplerFactory {
public:
	SamplerFactory(SamplerKind k, const ParameterGroup& params)
		: mKind(k)
		, mParams(params)
	{
	}
	uint32 requestedSampleCount() const override { return (uint32)mParams.getUInt("sample_count", DEF_SAMPLE_COUNT); }
	std::shared_ptr<ISampler> createInstance(uint32 sample_count, Random& rnd) const override
	{
		switch (mKind) {
		case SamplerKind::MJitt: {
			const uint32 PRIME = 14512081;
			// note: the seed default is evaluated even when 'seed' is given (argument of getUInt) -> always one draw
			const uint32 defSeed = PRIME ^ rnd.get32();
			return std::make_shared<MultiJitteredSampler>(sample_count, (uint32)mParams.getUInt("bins", std::max(1u, sample_count)),
														  (uint32)mParams.getUInt("seed", defSeed));
		}
		case SamplerKind::Sobol: return std::make_shared<SobolSampler>(rnd, sample_count);
		case SamplerKind::Stratified: return std::make_shared<StratifiedSampler>(sample_count, (uint32)mParams.getUInt("bins", std::max(1u, sample_count)));
		case SamplerKind::Uniform: return std::make_shared<UniformSampler>(sample_count);
		case SamplerKind::Halton: { // HaltonSamplerFactory::createInstance, HaltonSampler.cpp:135-141
			const uint32 bx = (uint32)mParams.getUInt("base_x", 13), by = (uint32)mParams.getUInt("base_y", 47);
			return std::make_shared<HaltonSampler>(sample_count, bx, by, (uint32)mParams.getUInt("burnin", std::max(bx, by)), false);
		}
		case SamplerKind::Hammersley: { // HammersleySamplerFactory::createInstance, :159-164
			const uint32 bx = (uint32)mParams.getUInt("base_x", 13);
			return std::make_shared<HaltonSampler>(sample_count, bx, 47, (uint32)mParams.getUInt("burnin", bx), true);
		}
		default: return std::make_shared<RandomSampler>(sample_count);
		}
	}

private:
	SamplerKind mKind;
	ParameterGroup mParams;
};
class SamplerPlugin : public ISamplerPlugin {
public:
	explicit SamplerPlugin(SamplerKind k)
		: mKind(k)
	{
	}
	std::shared_ptr<ISamplerFactory> create(const std::string&, const SceneLoadContext& ctx) override
	{
		if ((mKind == SamplerKind::Sobol || mKind == SamplerKind::Halton || mKind == SamplerKind::Hammersley) && ctx.environment()->renderSettings().progressive) {
			PR_LOG(L_WARNING) << "Sobol, halton and hammersley samplers do not support progressive rendering. Using 'mjitt' instead" << std::endl;
			return ctx.loadSamplerFactory("mjitt", ctx.parameters());
		}
		return std::make_shared<SamplerFactory>(mKind, ctx.parameters());
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> rnd({ "random" });
		static const std::vector<std::string> sob({ "sobol" });
		static const std::vector<std::string> mj({ "multijittered", "multi_jittered", "jittered", "multijitter", "multi_jitter", "jitter", "mjitt", "jitt" });
		static const std::vector<std::string> strat({ "stratified" });
		static const std::vector<std::string> uni({ "uniform" });
		static const std::vector<std::string> hal({ "halton" });
		static const std::vector<std::string> ham({ "hammersley" });
		switch (mKind) {
		case SamplerKind::Random: return rnd;
		case SamplerKind::Sobol: return sob;
		case SamplerKind::Stratified: return strat;
		case SamplerKind::Uniform: return uni;
		case SamplerKind::Halton: return hal;
		case SamplerKind::Hammersley: return ham;
		default: return mj;
		}
	}
	std::string specification(const std::string&) const override { return "Sampler: sample_count (128) [bins, seed for mjitt]"; }

private:
	SamplerKind mKind;
};

// ------------------------------------------------------------------ filters
// All tabulated pixel filters of the reference share one construction (plugins/main/filter/{Mitchell,Triangle,Gaussian,
// Lanczos}Filter.cpp): a radial profile sampled at integer pixel offsets of the first quadrant, normalised so that the
// mirrored (2r+1)^2 table sums to one.  Only the profile differs.
enum class FilterProfile { Mitchell, Triangle, Gaussian, Lanczos, Block };
static float filterProfile(FilterProfile kind, float r, int radius)
{ // r = distance in pixels
	switch (kind) {
	case FilterProfile::Mitchell: { // MitchellFilter.cpp: B = C = 1/3, argument 2 r / radius
		const float B = 1 / 3.0f, C = 1 / 3.0f;
		const float x = std::abs(2 * r / radius);
		if (x < 1)
			return ((12 - 9 * B - 6 * C) * x * x * x + (-18 + 12 * B + 6 * C) * x * x + (6 - 2 * B)) / 6;
		if (x < 2)
			return ((-B - 6 * C) * x * x * x + (6 * B + 30 * C) * x * x + (-12 * B - 48 * C) * x + (8 * B + 24 * C)) / 6;
		return 0.0f;
	}
	case FilterProfile::Triangle: // TriangleFilter.cpp:45
		return r <= radius ? 1 - r / (float)radius : 0.0f;
	case FilterProfile::Gaussian: { // GaussianFilter.cpp:40-46: variance 0.2 on the normalised distance
		const float x	  = r / (float)radius;
		const float alpha = 1 / (2 * 0.2f);
		return x <= 1.0f ? std::exp(-alpha * x * x) : 0.0f;
	}
	case FilterProfile::Lanczos: { // LanczosFilter.cpp:31-41
		auto sinc = [](float x) { return PR_INV_PI * std::sin(PR_PI * x) / x; };
		if (r <= PR_EPSILON)
			return 1.0f;
		return r <= radius ? sinc(r) * sinc(r / radius) : 0.0f;
	}
	default:
		return 1.0f;
	}
}
class TabulatedFilter : public IFilter {
public:
	TabulatedFilter(FilterProfile kind, int radius)
		: mRadius(radius)
	{
		if (mRadius == 0)
			return;
		const int half = mRadius + 1;
		mTable.assign(half * (size_t)half, 0.0f);
		// weights of the full table: centre once, axis entries twice, the rest four times
		float centre = 0, axes = 0, quadrant = 0;
		for (int y = 0; y < half; ++y)
			for (int x = 0; x < half; ++x) {
				const float w		 = filterProfile(kind, std::sqrt((float)(x * x + y * y)), mRadius);
				mTable[y * half + x] = w;
				(x == 0 && y == 0 ? centre : (x == 0 || y == 0 ? axes : quadrant)) += w;
			}
		const float norm = 1.0f / (centre + 2 * axes + 4 * quadrant);
		for (float& w : mTable)
			w *= norm;
	}
	int radius() const override { return mRadius; }
	float evalWeight(float x, float y) const override
	{
		if (mRadius == 0)
			return 1;
		// the reference clamps to mRadius+1 and indexes a (mRadius+1)^2 table with .at(); |x|,|y| <= mRadius here
		const int ix = std::min((int)std::round(std::abs(x)), mRadius);
		const int iy = std::min((int)std::round(std::abs(y)), mRadius);
		return mTable[iy * (mRadius + 1) + ix];
	}

private:
	int mRadius;
	std::vector<float> mTable;
};
class BlockFilter : public IFilter { // plugins/main/filter/BlockFilter.cpp: constant weight 1/(2r+1)^2
public:
	explicit BlockFilter(int radius)
		: mRadius(radius)
	{
	}
	int radius() const override { return mRadius; }
	float evalWeight(float, float) const override { return 1.0f / ((2 * mRadius + 1) * (2 * mRadius + 1)); }

private:
	int mRadius;
};
class FilterFactory : public IFilterFactory {
public:
	FilterFactory(FilterProfile kind, const ParameterGroup& p)
		: mKind(kind)
		, mParams(p)
	{
	}
	std::shared_ptr<IFilter> createInstance() const override
	{
		const int radius = (int)mParams.getInt("radius", 3);
		if (mKind == FilterProfile::Block)
			return std::make_shared<BlockFilter>(radius);
		return std::make_shared<TabulatedFilter>(mKind, radius);
	}

private:
	FilterProfile mKind;
	ParameterGroup mParams;
};
class FilterPlugin : public IFilterPlugin {
public:
	explicit FilterPlugin(FilterProfile kind)
		: mKind(kind)
	{
	}
	std::shared_ptr<IFilterFactory> create(const std::string&, const SceneLoadContext& ctx) override
	{
		return std::make_shared<FilterFactory>(mKind, ctx.parameters());
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names[] = { { "mitchell", "default" }, { "tri", "triangle" }, { "gaussian", "gauss" }, { "lanczos", "sinc", "lancz" },
														  { "block", "blur" } };
		return names[(int)mKind];
	}
	std::string specification(const std::string&) const override { return "Pixel filter: radius"; }

private:
	FilterProfile mKind;
};

// ------------------------------------------------------------------ spectral mappers
class RandomSpectralMapperFactory : public ISpectralMapperFactory { // spectralmapper/random.cpp
public:
	void describe(const SpectralMapperBuildInput&, prb_spectral_mapper& out, std::vector<float>&) override { out.type = PRB_MAPPER_RANDOM; }
};
class RandomSpectralMapperPlugin : public ISpectralMapperPlugin {
public:
	std::shared_ptr<ISpectralMapperFactory> create(const std::string&, const SceneLoadContext&) override { return std::make_shared<RandomSpectralMapperFactory>(); }
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "random" });
		return names;
	}
	std::string specification(const std::string&) const override { return "Random Spectral Mapper"; }
};

class CIESpectralMapperFactory : public ISpectralMapperFactory { // spectralmapper/cie.cpp:13-99, CIE::sample_(trunc_)xyz / _y (CIE.h:66-127)
public:
	explicit CIESpectralMapperFactory(bool onlyY)
		: mOnlyY(onlyY)
	{
	}
	void describe(const SpectralMapperBuildInput& in, prb_spectral_mapper& out, std::vector<float>& pool) override
	{
		const SpectralRange range = in.cameraRange;
		if (!(range.Start >= PR_CIE_WAVELENGTH_START && range.End <= PR_CIE_WAVELENGTH_END))
			throw std::runtime_error("cie spectral mapper: the camera range must lie inside the CIE range"); // createInstance returns nullptr
		// StaticCDF (src/base/math/Distribution1D.h:11-46): running sum of data / N in fp32, normalised, last entry forced to 1
		constexpr size_t N = PR_CIE_SAMPLE_COUNT;
		std::vector<float> cdf(N + 1);
		const float *X = CIE::table(0), *Y = CIE::table(1), *Z = CIE::table(2);
		cdf[0] = 0.0f;
		for (size_t i = 1; i < N + 1; ++i)
			cdf[i] = mOnlyY ? cdf[i - 1] + Y[i - 1] / N : cdf[i - 1] + (X[i - 1] + Y[i - 1] + Z[i - 1]) / N;
		if (cdf[N] < PR_EPSILON) {
			for (size_t i = 1; i < N + 1; ++i)
				cdf[i] = float(i) / float(N);
		} else {
			for (size_t i = 1; i < N + 1; ++i)
				cdf[i] /= cdf[N];
		}
		cdf[N] = 1.0f;
		const auto evalContinuous = [&](float x) { // Distribution1D::evalContinuous, Distribution1D.inl:106-112
			const size_t size = N + 1;
			const size_t off  = std::min<size_t>(size - 2, (size_t)(x * (size - 1)));
			const float dt	  = x * (size - 1) - off;
			return cdf[off] * (1 - dt) + cdf[off + 1] * dt;
		};
		out.type			= PRB_MAPPER_CIE;
		out.cdf_offset		= (uint32)pool.size();
		out.cdf_size		= (uint32)cdf.size();
		out.trunc_cdf_start = evalContinuous((range.Start - PR_CIE_WAVELENGTH_START) / PR_CIE_WAVELENGTH_RANGE);
		out.trunc_cdf_end	= evalContinuous((range.End - PR_CIE_WAVELENGTH_START) / PR_CIE_WAVELENGTH_RANGE);
		pool.insert(pool.end(), cdf.begin(), cdf.end());
	}

private:
	bool mOnlyY;
};
class CIESpectralMapperPlugin : public ISpectralMapperPlugin {
public:
	std::shared_ptr<ISpectralMapperFactory> create(const std::string& type_name, const SceneLoadContext& ctx) override
	{
		const bool onlyY = type_name == "cie_y" || type_name == "visible_y" || ctx.parameters().getBool("only_y", false);
		return std::make_shared<CIESpectralMapperFactory>(onlyY);
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "cie", "cie_y", "visible", "visible_y" });
		return names;
	}
	std::string specification(const std::string&) const override { return "CIE Spectral Mapper: only_y (bool, false)"; }
};

class AGHSpectralMapperFactory : public ISpectralMapperFactory { // spectralmapper/agh.cpp:14-155
public:
	explicit AGHSpectralMapperFactory(bool cmis)
		: mCMIS(cmis)
	{
	}
	void describe(const SpectralMapperBuildInput& in, prb_spectral_mapper& out, std::vector<float>&) override
	{
		constexpr float AStd = 0.0072f, BStd = 538;
		const auto single	= [&](float lambda) { return std::tanh(AStd * (BStd - lambda)); }; // aghSingle
		out.type			= mCMIS ? PRB_MAPPER_AGH_CMIS : PRB_MAPPER_AGH_HERO;
		out.trunc_cdf_start = single(in.cameraRange.Start);									 // mCameraC
		out.trunc_cdf_end	= single(in.cameraRange.Start) - single(in.cameraRange.End); // mCameraN
	}

private:
	bool mCMIS;
};
class AGHSpectralMapperPlugin : public ISpectralMapperPlugin {
public:
	std::shared_ptr<ISpectralMapperFactory> create(const std::string&, const SceneLoadContext& ctx) override
	{
		return std::make_shared<AGHSpectralMapperFactory>(ctx.parameters().getBool("cmis", true));
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "agh" });
		return names;
	}
	std::string specification(const std::string&) const override { return "AGH Spectral Mapper: cmis (bool, true)"; }
};

struct SPDParameters { // spd.cpp:161-176
	uint32 NumberOfBins			= (uint32)PR_CIE_WAVELENGTH_RANGE;
	int Method					= 2; // 0 none, 1 Y, 2 XYZ, 3 sRGB
	bool UseNormalizedLights	= true;
	bool EnsureCompleteSampling = true;
	uint32 SmoothIterations		= 0;
	bool UseCMIS				= true;
};
class SPDSpectralMapperFactory : public ISpectralMapperFactory { // spd.cpp:192-357 (pixel distribution)
public:
	explicit SPDSpectralMapperFactory(const SPDParameters& p)
		: mP(p)
	{
	}
	void describe(const SpectralMapperBuildInput& in, prb_spectral_mapper& out, std::vector<float>& pool) override
	{
		const uint32 bins = mP.NumberOfBins;
		std::vector<float> fullPower(bins, 0.0f), lightPower(bins, 0.0f);
		const SpectralRange range = in.cameraRange;
		const auto bin2wvl		  = [=](uint32 bin) { return range.Start + (bin / float(bins - 1)) * range.span(); };
		for (const Light& light : in.lightSampler->lights()) {
			// calcLightDistribution, spd.cpp:220-256
			for (uint32 i = 0; i < bins; i += 4) {
				const uint32 k = std::min<uint32>(bins - i, 4);
				SpectralBlob wavelengths = SpectralBlob::Zero();
				for (uint32 j = 0; j < k; ++j)
					wavelengths(j) = bin2wvl(i + j);
				for (uint32 j = k; j < 4; ++j)
					wavelengths(j) = wavelengths(0);
				const SpectralBlob output = light.averagePower(wavelengths);
				for (uint32 j = 0; j < k; ++j)
					lightPower[i + j] = output(j);
			}
			if (mP.UseNormalizedLights) {
				const float dt = 1.0f / (bins - 1);
				float integral = 0;
				for (float f : lightPower)
					integral += f * dt;
				if (integral > PR_EPSILON) {
					const float invnorm = 1 / integral;
					for (float& f : lightPower)
						f *= invnorm;
				}
			}
			for (uint32 i = 0; i < bins; ++i)
				fullPower[i] += lightPower[i];
		}
		// applyPostprocessing, spd.cpp:258-305
		int method = mP.Method;
		if (range.Start > PR_CIE_WAVELENGTH_END || range.End < PR_CIE_WAVELENGTH_START)
			method = 0;
		for (uint32 i = 0; i < bins; ++i) {
			const float w = bin2wvl(i);
			if (method == 1)
				fullPower[i] *= CIE::eval_y(w);
			else if (method == 2)
				fullPower[i] *= (CIE::eval_x(w) + CIE::eval_y(w) + CIE::eval_z(w));
			else if (method == 3) {
				const float X = CIE::eval_x(w), Y = CIE::eval_y(w), Z = CIE::eval_z(w); // RGBConverter::fromXYZ (sRGB D65)
				const float R = 3.240479f * X - 1.537150f * Y - 0.498535f * Z;
				const float G = -0.969256f * X + 1.875991f * Y + 0.041556f * Z;
				const float B = 0.055648f * X - 0.204043f * Y + 1.057311f * Z;
				fullPower[i] *= (R + G + B);
			}
		}
		for (uint32 it = 0; it < mP.SmoothIterations; ++it) {
			const std::vector<float> tmp = fullPower;
			for (size_t i = 0; i < tmp.size(); ++i) {
				const float prevM = (i == 0) ? tmp.front() : tmp[i - 1];
				const float nextM = (i == tmp.size() - 1) ? tmp.back() : tmp[i + 1];
				fullPower[i]	  = (prevM + tmp[i] + nextM) / 3;
			}
		}
		if (mP.EnsureCompleteSampling)
			for (float& f : fullPower)
				f = std::max(1e-2f, f);
		Distribution1D distr(bins);
		distr.generate([&](size_t bin) { return fullPower[bin]; });
		out.type	   = mP.UseCMIS ? PRB_MAPPER_SPD_CMIS : PRB_MAPPER_SPD_HERO;
		out.cdf_offset = (uint32)pool.size();
		out.cdf_size   = (uint32)distr.cdf().size();
		pool.insert(pool.end(), distr.cdf().begin(), distr.cdf().end());
	}

private:
	SPDParameters mP;
};
class SPDSpectralMapperPlugin : public ISpectralMapperPlugin {
public:
	std::shared_ptr<ISpectralMapperFactory> create(const std::string&, const SceneLoadContext& ctx) override
	{
		SPDParameters parameters;
		parameters.NumberOfBins = (uint32)ctx.parameters().getUInt("bins", parameters.NumberOfBins);
		std::string weighting	= ctx.parameters().getString("weighting", "xyz");
		std::transform(weighting.begin(), weighting.end(), weighting.begin(), ::tolower);
		if (weighting == "none")
			parameters.Method = 0;
		else if (weighting == "y")
			parameters.Method = 1;
		else if (weighting == "rgb" || weighting == "srgb")
			parameters.Method = 3;
		else
			parameters.Method = 2;
		parameters.EnsureCompleteSampling = ctx.parameters().getBool("complete", parameters.EnsureCompleteSampling);
		parameters.UseNormalizedLights	  = ctx.parameters().getBool("normalized", parameters.UseNormalizedLights);
		parameters.SmoothIterations		  = (uint32)ctx.parameters().getUInt("smooth_iterations", parameters.SmoothIterations);
		parameters.UseCMIS				  = ctx.parameters().getBool("cmis", parameters.UseCMIS);
		return std::make_shared<SPDSpectralMapperFactory>(parameters);
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "spd", "default" });
		return names;
	}
	std::string specification(const std::string&) const override
	{
		return "SPD Spectral Mapper: bins (440), weighting none|y|rgb|srgb|xyz (xyz), complete (true), normalized (true), smooth_iterations (0), cmis (true)";
	}
};
} // namespace

// ------------------------------------------------------------------ 'direct' integrator -> device
// reference plugins/main/integrators/direct.cpp:44-569.  IntDirectInstance::onTile forwards the tile to
// prb_render_tiles (include/prb200_abi.h) instead of walking rays on the CPU.
class IntDirectInstance : public IIntegratorInstance {
public:
	void onTile(RenderTileSession& session) override;
};
class IntDirect : public IIntegrator {
public:
	IntDirect(const DiParameters& p, bool power, bool emissiveScatter)
		: mParameters(p)
		, mPower(power)
		, mEmissiveScatter(emissiveScatter)
	{
	}
	std::shared_ptr<IIntegratorInstance> createThreadInstance(RenderContext*, size_t) override { return std::make_shared<IntDirectInstance>(); }
	void describe(prb_settings& s) const override
	{
		s.max_ray_depth		 = (uint32)mParameters.MaxCameraRayDepthHard;
		s.soft_max_ray_depth = (uint32)mParameters.MaxCameraRayDepthSoft;
		s.mis_power			 = mPower ? 1 : 0;
		s.do_nee			 = mParameters.DoNEE;
		s.do_direct			 = mParameters.DoDirect;
		s.emissive_scatter	 = mEmissiveScatter;
	}

private:
	DiParameters mParameters;
	bool mPower, mEmissiveScatter;
};
class IntDirectFactory : public IIntegratorFactory { // direct.cpp:498-538
public:
	explicit IntDirectFactory(const ParameterGroup& params)
	{
		mParameters.MaxCameraRayDepthHard = (size_t)params.getUInt("max_ray_depth", mParameters.MaxCameraRayDepthHard);
		mParameters.MaxCameraRayDepthSoft = std::min(mParameters.MaxCameraRayDepthHard, (size_t)params.getUInt("soft_max_ray_depth", mParameters.MaxCameraRayDepthSoft));
		std::string mode				  = params.getString("mis", "balance");
		std::transform(mode.begin(), mode.end(), mode.begin(), ::tolower);
		mPower				 = mode == "power";
		mParameters.DoNEE	 = params.getBool("nee", true);
		mParameters.DoDirect = params.getBool("direct", true);
		mEmissiveScatter	 = params.getBool("emissive_scatter", true);
	}
	std::shared_ptr<IIntegrator> createInstance() const override { return std::make_shared<IntDirect>(mParameters, mPower, mEmissiveScatter); }

private:
	DiParameters mParameters;
	bool mPower = false, mEmissiveScatter = true;
};
class IntDirectFactoryFactory : public IIntegratorPlugin {
public:
	std::shared_ptr<IIntegratorFactory> create(const std::string&, const SceneLoadContext& ctx) override { return std::make_shared<IntDirectFactory>(ctx.parameters()); }
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "direct", "standard", "default" });
		return names;
	}
	std::string specification(const std::string&) const override
	{
		return "PT / Unidirectional Path Tracing: max_ray_depth (64), soft_max_ray_depth (4), mis balance|power, nee (true), direct (true), emissive_scatter (true)";
	}
};

void IntDirectInstance::onTile(RenderTileSession& session)
{
	const RenderTile* t = session.tile();
	prb_tile pt{ t->sx, t->sy, t->ex, t->ey };
	const prb_status st = prb_render_tiles(session.context()->deviceContext(), &pt, 1, session.iteration(), 1);
	if (st != PRB_OK)
		PR_LOG(L_ERROR) << "prb_render_tiles failed: " << prb_last_error() << std::endl;
}

// ------------------------------------------------------------------ 'ao' integrator -> device
// reference plugins/main/integrators/ao.cpp: one parameter, sample_count (occlusion rays per pixel sample, default 10).  The
// tiles go to prb_render_tiles like 'direct'; RenderContext selects the kernels with prb_set_integrator.
class IntAO : public IIntegrator {
public:
	explicit IntAO(uint32 sampleCount)
		: mSampleCount(sampleCount)
	{
	}
	std::shared_ptr<IIntegratorInstance> createThreadInstance(RenderContext*, size_t) override { return std::make_shared<IntDirectInstance>(); }
	void describe(prb_settings& s) const override
	{ // no path beyond the first hit, no light sampling
		s.max_ray_depth		 = 1;
		s.soft_max_ray_depth = 1;
		s.do_nee = s.do_direct = s.emissive_scatter = 0;
	}
	prb_integrator deviceIntegrator() const override { return prb_integrator{ PRB_INTEGRATOR_AO, mSampleCount }; }

private:
	uint32 mSampleCount;
};
class IntAOFactory : public IIntegratorFactory {
public:
	explicit IntAOFactory(const ParameterGroup& params)
	{
		const uint64 n = params.getUInt("sample_count", 10);
		if (n == 0)
			PR_LOG(L_ERROR) << "[ao] sample_count must be at least 1; using 1" << std::endl;
		mSampleCount = (uint32)std::min<uint64>(std::max<uint64>(n, 1), 0xFFFFFFFFu);
	}
	std::shared_ptr<IIntegrator> createInstance() const override { return std::make_shared<IntAO>(mSampleCount); }

private:
	uint32 mSampleCount = 10;
};
class IntAOFactoryFactory : public IIntegratorPlugin {
public:
	std::shared_ptr<IIntegratorFactory> create(const std::string&, const SceneLoadContext& ctx) override { return std::make_shared<IntAOFactory>(ctx.parameters()); }
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "ao", "ambientocclusion", "occlusion" });
		return names;
	}
	std::string specification(const std::string&) const override { return "AO / Ambient Occlusion: sample_count (10)"; }
};

// ------------------------------------------------------------------ 'visualfeedback' integrator -> device
// reference plugins/main/integrators/visualfeedback.cpp: one parameter, mode (what the colour of a pixel shows, default
// colored_entity_id; the names are listed in vfModeNames).  The tiles go to prb_render_tiles like 'direct'; RenderContext
// selects the kernel with prb_set_integrator.
static const char* const vfModeNames[PRB_VF__COUNT] = { "colored_entity_id", "colored_material_id", "colored_emission_id",
														 "colored_primitive_id", "parameter", "inside", "ndotv" }; // PRB_VF_*
class IntVF : public IIntegrator {
public:
	explicit IntVF(uint32 mode)
		: mMode(mode)
	{
	}
	std::shared_ptr<IIntegratorInstance> createThreadInstance(RenderContext*, size_t) override { return std::make_shared<IntDirectInstance>(); }
	void describe(prb_settings& s) const override
	{ // no path beyond the first hit, no light sampling
		s.max_ray_depth		 = 1;
		s.soft_max_ray_depth = 1;
		s.do_nee = s.do_direct = s.emissive_scatter = 0;
	}
	prb_integrator deviceIntegrator() const override
	{
		prb_integrator r{};
		r.type = PRB_INTEGRATOR_VF;
		r.mode = mMode;
		return r;
	}

private:
	uint32 mMode;
};
class IntVFFactory : public IIntegratorFactory {
public:
	explicit IntVFFactory(uint32 mode)
		: mMode(mode)
	{
	}
	std::shared_ptr<IIntegrator> createInstance() const override { return std::make_shared<IntVF>(mMode); }

private:
	uint32 mMode;
};
class IntVFFactoryFactory : public IIntegratorPlugin {
public:
	std::shared_ptr<IIntegratorFactory> create(const std::string&, const SceneLoadContext& ctx) override
	{
		std::string mode = ctx.parameters().getString("mode", vfModeNames[PRB_VF_ENTITY_ID]);
		std::transform(mode.begin(), mode.end(), mode.begin(), ::tolower);
		for (uint32 m = 0; m < PRB_VF__COUNT; ++m)
			if (mode == vfModeNames[m])
				return std::make_shared<IntVFFactory>(m);
		PR_LOG(L_ERROR) << "[visualfeedback] Unknown mode " << mode << std::endl;
		return nullptr;
	}
	const std::vector<std::string>& getNames() const override
	{
		static const std::vector<std::string> names({ "visualfeedback", "vf" });
		return names;
	}
	std::string specification(const std::string&) const override
	{
		return "VF / Visual Feedback: mode colored_entity_id|colored_material_id|colored_emission_id|colored_primitive_id|parameter|inside|ndotv (colored_entity_id)";
	}
};

void registerScenePlugins(std::vector<std::shared_ptr<IPlugin>>& out)
{
	out.push_back(std::make_shared<MeshEntityPlugin>());
	out.push_back(std::make_shared<SphereEntityPlugin>());
	out.push_back(std::make_shared<PlaneEntityPlugin>());
	out.push_back(std::make_shared<PerspectiveCameraPlugin>());
	out.push_back(std::make_shared<OrthoCameraPlugin>());
	out.push_back(std::make_shared<DiffuseEmissionPlugin>());
	out.push_back(std::make_shared<EnvironmentLightFactory>());
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Sobol));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::MJitt));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Random));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Stratified));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Uniform));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Halton));
	out.push_back(std::make_shared<SamplerPlugin>(SamplerKind::Hammersley));
	for (FilterProfile k : { FilterProfile::Mitchell, FilterProfile::Triangle, FilterProfile::Gaussian, FilterProfile::Lanczos, FilterProfile::Block })
		out.push_back(std::make_shared<FilterPlugin>(k));
	out.push_back(std::make_shared<SPDSpectralMapperPlugin>());
	out.push_back(std::make_shared<RandomSpectralMapperPlugin>());
	out.push_back(std::make_shared<CIESpectralMapperPlugin>());
	out.push_back(std::make_shared<AGHSpectralMapperPlugin>());
	out.push_back(std::make_shared<IntDirectFactoryFactory>());
	out.push_back(std::make_shared<IntAOFactoryFactory>());
	out.push_back(std::make_shared<IntVFFactoryFactory>());
}
} // namespace PR
