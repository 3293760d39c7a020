// Host-side mirror of the PearRay interfaces that sit on the spectral path-tracing hot path.
// Same names, argument meaning and error behaviour as the reference (file:line cited per class);
// the objects do not execute the path on the CPU -- they describe themselves into the POD scene
// descriptor of include/prb200_abi.h, which the CUDA library consumes.
#pragma once
#include "datalisp.h"
#include "prh_math.h"
#include "../../include/prb200_abi.h"

#include <functional>
#include <iostream>
#include <map>
#include <memory>
#include <optional>
#include <string>
#include <unordered_map>
#include <vector>

namespace PR {
// ------------------------------------------------------------------ logging (reference src/base/Logger.h)
enum LogLevel { L_DEBUG = 0, L_INFO, L_WARNING, L_ERROR, L_FATAL };
int& logVerbosity(); // messages below this level are dropped (default L_WARNING)
std::ostream& logStream(LogLevel lvl);
#define PR_LOG(l) ::PR::logStream(::PR::l)

// ------------------------------------------------------------------ parameters
// reference src/loader/parameter/Parameter.h, ParameterGroup.h
enum class ParameterType { Invalid = 0, Bool, Int, UInt, Number, String, Reference };
constexpr uint32 P_INVALID_REFERENCE = 0xFFFFFFFFu;

class Parameter {
public:
	Parameter() = default;
	static Parameter fromBool(bool v);
	static Parameter fromInt(int64 v);
	static Parameter fromUInt(uint64 v);
	static Parameter fromNumber(float v);
	static Parameter fromString(const std::string& v);
	static Parameter fromReference(uint32 id);
	static Parameter fromBoolArray(const std::vector<bool>& v);
	static Parameter fromIntArray(const std::vector<int64>& v);
	static Parameter fromNumberArray(const std::vector<float>& v);
	static Parameter fromStringArray(const std::vector<std::string>& v);

	ParameterType type() const { return mType; }
	bool isValid() const { return mType != ParameterType::Invalid; }
	bool isArray() const { return mIsArray; }
	size_t arraySize() const;
	bool getBool(bool def) const;
	int64 getInt(int64 def) const;
	uint64 getUInt(uint64 def) const;
	float getNumber(float def) const; // Int/UInt/Number all convert
	float getNumber(size_t idx, float def) const;
	std::string getString(const std::string& def) const;
	std::string getString(size_t idx, const std::string& def) const;
	uint32 getReference() const { return mType == ParameterType::Reference ? (uint32)mInts.at(0) : P_INVALID_REFERENCE; }

private:
	ParameterType mType = ParameterType::Invalid;
	bool mIsArray		= false;
	std::vector<int64> mInts;
	std::vector<float> mNumbers;
	std::vector<std::string> mStrings;
};

class ParameterGroup {
public:
	void addParameter(const std::string& name, const Parameter& p) { mNamed[name] = p; }
	void addParameter(const Parameter& p) { mPositional.push_back(p); }
	bool hasParameter(const std::string& name) const { return mNamed.count(name) > 0; }
	Parameter getParameter(const std::string& name) const
	{
		auto it = mNamed.find(name);
		return it == mNamed.end() ? Parameter() : it->second;
	}
	Parameter getParameter(size_t idx) const { return idx < mPositional.size() ? mPositional[idx] : Parameter(); }
	size_t positionalParameterCount() const { return mPositional.size(); }
	bool getBool(const std::string& n, bool def) const { return getParameter(n).getBool(def); }
	int64 getInt(const std::string& n, int64 def) const { return getParameter(n).getInt(def); }
	uint64 getUInt(const std::string& n, uint64 def) const { return getParameter(n).getUInt(def); }
	float getNumber(const std::string& n, float def) const { return getParameter(n).getNumber(def); }
	std::string getString(const std::string& n, const std::string& def) const { return getParameter(n).getString(def); }
	std::string getString(size_t idx, const std::string& def) const { return getParameter(idx).getString(def); }
	Vector3f getVector3f(const std::string& n, const Vector3f& def) const;

private:
	std::map<std::string, Parameter> mNamed;
	std::vector<Parameter> mPositional;
};

// ------------------------------------------------------------------ spectral helpers
struct SpectralRange { // reference src/core/spectral/SpectralRange.h
	float Start = -1, End = -1;
	SpectralRange() = default;
	SpectralRange(float s, float e)
		: Start(s)
		, End(e)
	{
	}
	float span() const { return End - Start; }
	bool isStartUnbounded() const { return Start < 0; }
	bool isEndUnbounded() const { return End < 0; }
	SpectralRange bounded(const SpectralRange& o) const { return SpectralRange(isStartUnbounded() ? o.Start : Start, isEndUnbounded() ? o.End : End); }
	SpectralRange& operator+=(const SpectralRange& o)
	{
		Start = isStartUnbounded() ? o.Start : (o.isStartUnbounded() ? Start : std::min(Start, o.Start));
		End	  = std::max(End, o.End);
		return *this;
	}
	SpectralRange operator+(const SpectralRange& o) const
	{
		SpectralRange t = *this;
		t += o;
		return t;
	}
};

constexpr int PR_CIE_SAMPLE_COUNT		= 441; // reference src/core/spectral/CIE.h:18-29 (CIE 2006)
constexpr float PR_CIE_WAVELENGTH_START = 390;
constexpr float PR_CIE_WAVELENGTH_END	= 830;
constexpr float PR_CIE_Y_NORM_SUM		= 113.042314572337f;
constexpr float PR_CIE_WAVELENGTH_RANGE = PR_CIE_WAVELENGTH_END - PR_CIE_WAVELENGTH_START;
constexpr float PR_CIE_WAVELENGTH_DELTA = PR_CIE_WAVELENGTH_RANGE / (PR_CIE_SAMPLE_COUNT - 1);
constexpr float PR_CIE_Y_NORM			= PR_CIE_Y_NORM_SUM * PR_CIE_WAVELENGTH_DELTA;

namespace CIE { // reference CIE::eval_x/y/z, src/core/spectral/CIE.h:41-58
float eval_x(float wavelength);
float eval_y(float wavelength);
float eval_z(float wavelength);
const float* table(int channel); // 0 x, 1 y, 2 z; PR_CIE_SAMPLE_COUNT entries
}

// reference EquidistantSpectrumView::lookup, src/core/spectral/EquidistantSpectrum.inl:34-41
float equidistantLookup(const float* data, size_t count, float start, float end, float wavelength);

class Distribution1D { // reference src/base/math/Distribution1D.inl
public:
	explicit Distribution1D(size_t size = 0)
		: mCDF(size + 1)
	{
	}
	size_t numberOfValues() const { return mCDF.size() - 1; }
	void generate(const std::function<float(size_t)>& f, float* sum = nullptr);
	float discretePdf(size_t x) const { return mCDF[x + 1] - mCDF[x]; }
	size_t sampleDiscrete(float u, float& pdf, float* rem = nullptr) const;
	float sampleContinuous(float u, float& pdf) const;
	const std::vector<float>& cdf() const { return mCDF; }

private:
	std::vector<float> mCDF;
};

// Jakob-Hanika RGB -> sigmoid coefficients; reference src/core/spectral/SpectralUpsampler.cpp:78-146
class SpectralUpsampler {
public:
	explicit SpectralUpsampler(const std::string& file); // pearray_b200/data/rgb2spec_srgb.bin
	void prepare(const float* r, const float* g, const float* b, float* out_a, float* out_b, float* out_c, size_t elems) const;
	uint32 resolution() const { return mRes; }
	const std::vector<float>& scale() const { return mScale; }
	const std::vector<float>& data() const { return mData; }
	static void computeSingle(float a, float b, float c, const float* wavelengths, float* out_weights, size_t elems);

private:
	uint32 mRes = 0;
	std::vector<float> mScale, mData;
};

// pcg32_fast; reference src/core/Random.h:26-179 + src/core/random/pcg_random.hpp (mcg_xsh_rs_64_32)
class Random {
public:
	explicit Random(uint64 seed = 4203893)
		: mState(seed | 3u)
	{
	}
	static constexpr uint64 MULT = 6364136223846793005ULL;
	uint32 get32()
	{
		const uint64 old = mState;
		mState			 = old * MULT;
		const uint32 rs	 = (uint32)(old >> 61);
		const uint64 x	 = old ^ (old >> 22);
		return (uint32)(x >> (22 + rs));
	}
	uint64 get64() { return ((uint64)get32() << 32) + get32(); } // libstdc++ uniform_int_distribution<uint64> over a 32-bit URNG
	uint32 get32(uint32 start, uint32 end);						 // [start, end-1], libstdc++ (>= 9) Lemire nearly-divisionless
	uint64 get64(uint64 start, uint64 end);						 // [start, end-1], libstdc++ 128-bit Lemire over get64()
	static float uint32ToFloat(uint32 v)
	{
		const uint32 u = (v >> 9) | 0x3F800000u;
		float f;
		std::memcpy(&f, &u, 4);
		return f - 1.0f;
	}
	static double uint64ToDouble(uint64 v)
	{
		const uint64 u = (v >> 12) | 0x3FF0000000000000ULL;
		double f;
		std::memcpy(&f, &u, 8);
		return f - 1.0;
	}
	float getFloat() { return uint32ToFloat(get32()); }
	// GCC evaluates the two unsequenced getFloat() arguments of Vector2f(getFloat(), getFloat()) right to left
	// (SURVEY F10): the FIRST draw becomes y, the second x.
	Vector2f get2D()
	{
		const float y = getFloat();
		const float x = getFloat();
		return Vector2f(x, y);
	}
	void advance(uint64 delta); // jump ahead by delta get32() calls
	uint64 state() const { return mState; }
	void setState(uint64 s) { mState = s; }

private:
	uint64 mState;
};
// std::shuffle(first,last,Random&) as libstdc++ 13 implements it for a 64-bit URBG (pairs of swaps)
void libstdcxxShuffle(std::vector<uint32>& perm, Random& rnd);

// ------------------------------------------------------------------ shading nodes
struct ShadingContext { // reference src/core/shader/ShadingContext.h
	Vector2f UV;
	SpectralBlob WavelengthNM;
};
enum class NodeType { FloatScalar, FloatSpectral, FloatVector };
enum NodeFlag : uint32 { NF_Const = 0x1, NF_SpectralVarying = 0x2, NF_TextureVarying = 0x4, NF_TimeVarying = 0x8 };

class NodeEmitter;
class INode { // reference src/core/shader/INode.h
public:
	INode(NodeType t, uint32 flags)
		: mType(t)
		, mFlags(flags)
	{
	}
	virtual ~INode() = default;
	NodeType type() const { return mType; }
	uint32 flags() const { return mFlags; }
	bool isSpectralVarying() const { return mFlags & NF_SpectralVarying; }
	virtual std::string dumpInformation() const = 0;

private:
	NodeType mType;
	uint32 mFlags;
};
class FloatScalarNode : public INode {
public:
	explicit FloatScalarNode(uint32 flags)
		: INode(NodeType::FloatScalar, flags)
	{
	}
	virtual float eval(const ShadingContext&) const = 0;
	virtual bool isConst() const { return false; }
};
class FloatSpectralNode : public INode {
public:
	explicit FloatSpectralNode(uint32 flags)
		: INode(NodeType::FloatSpectral, flags)
	{
	}
	virtual SpectralBlob eval(const ShadingContext&) const = 0;
	virtual SpectralRange spectralRange() const { return SpectralRange(); }
	// INode::queryRecommendedSize (image nodes: the image size; everything else 1 x 1)
	virtual void queryRecommendedSize(int& w, int& h) const { w = h = 1; }
	// flatten into the device node table, returns node id
	virtual uint32 emit(NodeEmitter& e) const = 0;
};
class NodeEmitter {
public:
	std::vector<prb_node> nodes;
	std::vector<float>* pool = nullptr;
	// set by the first image node that is emitted: the scene needs the RGB -> spectrum coefficient cube in its pool
	const SpectralUpsampler* upsampler = nullptr;
	uint32 add(const FloatSpectralNode* key, const prb_node& n);
	bool find(const FloatSpectralNode* key, uint32& id) const;
	uint32 emitNode(const std::shared_ptr<FloatSpectralNode>& n) { return n->emit(*this); }

private:
	std::unordered_map<const FloatSpectralNode*, uint32> mCache;
};
namespace NodeUtils { // reference src/core/shader/NodeUtils.cpp (32x32 UV average)
SpectralBlob average(const SpectralBlob& wvls, const FloatSpectralNode* node);
}
std::shared_ptr<FloatScalarNode> makeConstScalarNode(float f);
// NonParametricImageNode over an image file (plugins_nodes.cpp); interp: PRB_TEX_*, wraps: PRB_WRAP_*; null when unreadable
std::shared_ptr<FloatSpectralNode> makeImageNode(const std::string& file, int interp, int wrapS, int wrapT, const std::shared_ptr<SpectralUpsampler>& upsampler);
std::shared_ptr<FloatSpectralNode> makeConstSpectralNode(float f);

// ------------------------------------------------------------------ scene objects
class SceneCompiler;
class RenderTileSession;

enum MaterialSampleFlag : uint32 { // reference src/core/material/MaterialType.h
	MSF_Null			  = 0x1,
	MSF_DeltaDistribution = 0x2,
	MSF_SpectralVarying	  = 0x4,
	MSF_SpatialVarying	  = 0x8,
	MSF_TimeVarying		  = 0x10,
	MSF_Fluorescent		  = 0x20
};
enum class MaterialScatteringType : uint32 { DiffuseReflection = 0, SpecularReflection, DiffuseTransmission, SpecularTransmission };

struct MaterialEvalInput { // shading-space subset of reference MaterialEvalContext
	Vector3f V, L;
	SpectralBlob WavelengthNM;
	Vector2f UV;
	uint32 RayFlags = 0;
};
struct MaterialEvalOutput {
	SpectralBlob Weight, PDF_S;
	uint32 Flags = 0;
	MaterialScatteringType Type = MaterialScatteringType::DiffuseReflection;
};
struct MaterialSampleInput {
	Vector3f V;
	SpectralBlob WavelengthNM;
	Vector2f UV;
	uint32 RayFlags = 0;
	Random* RND		= nullptr;
};
struct MaterialSampleOutput {
	Vector3f L;
	SpectralBlob IntegralWeight, PDF_S;
	uint32 Flags				= 0;
	MaterialScatteringType Type = MaterialScatteringType::DiffuseReflection;
	bool isDelta() const { return Flags & MSF_DeltaDistribution; }
	bool isHeroCollapsing() const { return (Flags & MSF_DeltaDistribution) && (Flags & MSF_SpectralVarying); }
};

class IMaterial { // reference src/core/material/IMaterial.h:15-55
public:
	virtual ~IMaterial() = default;
	virtual bool hasOnlyDeltaDistribution() const { return false; }
	virtual std::string dumpInformation() const = 0;
	virtual void describe(prb_material& out, NodeEmitter& e) const = 0;
	// eval / sample run on the device through the session's context (prb_material_eval / _sample)
	void eval(const MaterialEvalInput& in, MaterialEvalOutput& out, const RenderTileSession& session) const;
	void sample(const MaterialSampleInput& in, MaterialSampleOutput& out, const RenderTileSession& session) const;
	uint32 id() const { return mID; }
	void setID(uint32 id) { mID = id; }

private:
	uint32 mID = PR_INVALID_ID;
};

class IEmission { // reference src/core/emission/IEmission.h:10-32
public:
	virtual ~IEmission() = default;
	virtual SpectralBlob power(const SpectralBlob& wvl) const = 0;
	virtual SpectralRange spectralRange() const				  = 0;
	virtual void describe(prb_emission& out, NodeEmitter& e) const = 0;
	virtual std::string dumpInformation() const = 0;
};

class ITransformable { // reference src/core/entity/ITransformable.h/.cpp
public:
	ITransformable(const std::string& name, const Transformf& t);
	virtual ~ITransformable() = default;
	const std::string& name() const { return mName; }
	const Transformf& transform() const { return mTransform; }
	const Transformf& invTransform() const { return mInvTransformCache; }
	const Matrix3f& normalMatrix() const { return mNormalMatrixCache; }
	const Matrix3f& invNormalMatrix() const { return mInvNormalMatrixCache; }
	float volumeScalefactor() const { return mJacobianDeterminant; }

private:
	std::string mName;
	Transformf mTransform, mInvTransformCache;
	Matrix3f mNormalMatrixCache, mInvNormalMatrixCache;
	float mJacobianDeterminant;
};

class MeshBase { // reference src/core/mesh/MeshBase.h (triangle/quad soup with shared indices)
public:
	std::string name;
	std::vector<float> vertices, normals, uvs;
	std::vector<uint32> indices;	  // 4 per face, PRB_INVALID_ID in 4th slot for triangles
	std::vector<uint32> materialSlots; // per face (may be empty -> 0)
	size_t faceCount() const { return indices.size() / 4; }
	size_t vertexCount() const { return vertices.size() / 3; }
	bool hasNormals() const { return !normals.empty(); }
	bool hasUVs() const { return !uvs.empty(); }
	bool isQuad(size_t f) const { return indices[f * 4 + 3] != PR_INVALID_ID; }
	Vector3f vertex(uint32 i) const { return { vertices[3 * i], vertices[3 * i + 1], vertices[3 * i + 2] }; }
	float faceArea(size_t f) const;					  // Face::surfaceArea, src/core/geometry/Face.h:62-68
	float surfaceArea(const Transformf& t) const;	  // MeshBase::surfaceArea(transform)
	BoundingBox constructBoundingBox() const;
	bool isValid(std::string* err) const;
};

class IEntity : public ITransformable { // reference src/core/entity/IEntity.h:52-107
public:
	IEntity(uint32 emission_id, const std::string& name, const Transformf& t)
		: ITransformable(name, t)
		, mVisibilityFlags(0x0F)
		, mEmissionID(emission_id)
	{
	}
	virtual std::string type() const							 = 0;
	virtual float localSurfaceArea() const						 = 0;
	virtual float worldSurfaceArea() const { return volumeScalefactor() * localSurfaceArea(); }
	virtual BoundingBox worldBoundingBox() const				 = 0;
	virtual float sampleParameterPointPDF() const { return 1.0f / worldSurfaceArea(); }
	virtual void describe(prb_entity& out, SceneCompiler& c) const = 0;
	bool hasEmission() const { return mEmissionID != PR_INVALID_ID; }
	uint32 emissionID() const { return mEmissionID; }
	uint32 visibilityFlags() const { return mVisibilityFlags; }
	void setVisibilityFlags(uint32 f) { mVisibilityFlags = f; }

private:
	uint32 mVisibilityFlags;
	uint32 mEmissionID;
};

class ICamera : public ITransformable { // reference src/core/camera/ICamera.h
public:
	using ITransformable::ITransformable;
	virtual std::string type() const			   = 0;
	virtual void describe(prb_camera& out) const = 0;
};

class IInfiniteLight : public ITransformable { // reference src/core/infinitelight/IInfiniteLight.h
public:
	using ITransformable::ITransformable;
	virtual bool hasDeltaDistribution() const { return false; }
	virtual SpectralBlob power(const SpectralBlob& wvl) const = 0;
	virtual SpectralRange spectralRange() const				  = 0;
	virtual void describe(prb_light& out, NodeEmitter& e) const = 0;
};

class ISampler { // reference src/core/sampler/ISampler.h:6-23
public:
	explicit ISampler(uint32 samples)
		: mMaxSamples(samples)
	{
	}
	virtual ~ISampler() = default;
	uint32 maxSamples() const { return mMaxSamples; }
	virtual float generate1D(Random& rnd, uint32 index)	   = 0;
	virtual Vector2f generate2D(Random& rnd, uint32 index) = 0;
	virtual void describe(prb_sampler& out, std::vector<float>& pool) const = 0;

private:
	uint32 mMaxSamples;
};
class ISamplerFactory {
public:
	virtual ~ISamplerFactory()												 = default;
	virtual uint32 requestedSampleCount() const								 = 0;
	virtual std::shared_ptr<ISampler> createInstance(uint32 sample_count, Random& rnd) const = 0;
};

class IFilter { // reference src/core/filter/IFilter.h
public:
	virtual ~IFilter()								   = default;
	virtual int radius() const						   = 0;
	virtual float evalWeight(float x, float y) const = 0;
};
class IFilterFactory {
public:
	virtual ~IFilterFactory()									  = default;
	virtual std::shared_ptr<IFilter> createInstance() const = 0;
};

class RenderContext;
class LightSampler;
struct SpectralMapperBuildInput {
	SpectralRange cameraRange, lightRange;
	const LightSampler* lightSampler = nullptr;
};
class ISpectralMapperFactory { // reference src/core/spectral/ISpectralMapperFactory.h; describe() builds the distribution
public:
	virtual ~ISpectralMapperFactory() = default;
	virtual void describe(const SpectralMapperBuildInput& in, prb_spectral_mapper& out, std::vector<float>& pool) = 0;
};

struct DiParameters { // reference direct.cpp:34-39
	size_t MaxCameraRayDepthHard = 64;
	size_t MaxCameraRayDepthSoft = 4;
	bool DoNEE					 = true;
	bool DoDirect				 = true;
};
class IIntegratorInstance { // reference src/core/integrator/IIntegrator.h:11-22
public:
	virtual ~IIntegratorInstance() = default;
	virtual void onStart() {}
	virtual void onEnd() {}
	virtual void onTile(RenderTileSession& session) = 0;
};
class IIntegrator { // reference src/core/integrator/IIntegrator.h:24-37
public:
	virtual ~IIntegrator() = default;
	virtual void onInit(RenderContext*) {}
	virtual void onStart() {}
	virtual void onEnd() {}
	virtual std::shared_ptr<IIntegratorInstance> createThreadInstance(RenderContext* ctx, size_t thread_index) = 0;
	virtual void describe(prb_settings& s) const = 0;
	// the record prb_set_integrator takes for this integrator (RenderContext applies it after prb_upload_scene)
	virtual prb_integrator deviceIntegrator() const { return prb_integrator{ PRB_INTEGRATOR_DIRECT, 0 }; }
};
class IIntegratorFactory { // reference src/core/integrator/IIntegratorFactory.h:7-12
public:
	virtual ~IIntegratorFactory()									 = default;
	virtual std::shared_ptr<IIntegrator> createInstance() const = 0;
};

// ------------------------------------------------------------------ plugins
// reference src/loader/plugin/Plugin.h:26-66, PluginManager.cpp
enum class PluginType { Camera, Emission, Entity, Filter, InfiniteLight, Integrator, Material, Node, Sampler, SpectralMapper };
class SceneLoadContext;
class IPlugin {
public:
	virtual ~IPlugin()				   = default;
	virtual PluginType type() const = 0;
	virtual const std::vector<std::string>& getNames() const = 0;
	virtual std::string specification(const std::string& type_name) const = 0; // human readable parameter list
};
template <typename T, PluginType PT>
class ITypedPlugin : public IPlugin {
public:
	PluginType type() const override { return PT; }
	virtual std::shared_ptr<T> create(const std::string& type_name, const SceneLoadContext& ctx) = 0;
};
using ICameraPlugin			= ITypedPlugin<ICamera, PluginType::Camera>;
using IEmissionPlugin		= ITypedPlugin<IEmission, PluginType::Emission>;
using IEntityPlugin			= ITypedPlugin<IEntity, PluginType::Entity>;
using IFilterPlugin			= ITypedPlugin<IFilterFactory, PluginType::Filter>;
using IInfiniteLightPlugin	= ITypedPlugin<IInfiniteLight, PluginType::InfiniteLight>;
using IIntegratorPlugin		= ITypedPlugin<IIntegratorFactory, PluginType::Integrator>;
using IMaterialPlugin		= ITypedPlugin<IMaterial, PluginType::Material>;
using INodePlugin			= ITypedPlugin<INode, PluginType::Node>;
using ISamplerPlugin		= ITypedPlugin<ISamplerFactory, PluginType::Sampler>;
using ISpectralMapperPlugin = ITypedPlugin<ISpectralMapperFactory, PluginType::SpectralMapper>;

#define PR_PLUGIN_API_VERSION 1
struct PluginInterface { // exported as extern "C" _pr_exports by external plugin objects
	int APIVersion;
	const char* FileName;
	const char* ClassName;
	const char* PluginName;
	const char* PluginVersion;
	IPlugin* (*InitFunction)();
};

template <typename PluginT>
class AbstractManager { // reference src/loader/plugin/AbstractManager.h:18-34 (first registration of a name wins)
public:
	void addFactory(const std::shared_ptr<PluginT>& p)
	{
		for (const auto& n : p->getNames())
			if (!mFactories.count(n))
				mFactories[n] = p;
	}
	std::shared_ptr<PluginT> getFactory(const std::string& name) const
	{
		auto it = mFactories.find(name);
		return it == mFactories.end() ? nullptr : it->second;
	}
	bool hasFactory(const std::string& n) const { return mFactories.count(n) > 0; }
	std::vector<std::string> names() const
	{
		std::vector<std::string> r;
		for (const auto& kv : mFactories)
			r.push_back(kv.first);
		return r;
	}

private:
	std::map<std::string, std::shared_ptr<PluginT>> mFactories;
};

class PluginManager { // reference src/loader/plugin/PluginManager.cpp:14-225
public:
	explicit PluginManager(const std::string& pluginPath = "");
	~PluginManager();
	bool tryLoad(const std::string& path); // dlopen, "_pr_exports", API version check
	void loadEmbeddedPlugins();
	const std::vector<std::shared_ptr<IPlugin>>& plugins() const { return mPlugins; }

private:
	std::vector<std::shared_ptr<IPlugin>> mPlugins;
	std::vector<void*> mLibraries;
};
void registerEmbeddedPlugins(std::vector<std::shared_ptr<IPlugin>>& out); // plugins_*.cpp

// ------------------------------------------------------------------ scene database / settings / environment
template <typename T>
class AbstractDatabase { // reference src/core/AbstractDatabase.h
public:
	uint32 add(const std::shared_ptr<T>& o)
	{
		mObjects.push_back(o);
		return (uint32)mObjects.size() - 1;
	}
	uint32 add(const std::string& name, const std::shared_ptr<T>& o)
	{
		const uint32 id = add(o);
		mNamed[name]	= id;
		return id;
	}
	bool has(const std::string& n) const { return mNamed.count(n) > 0; }
	uint32 getID(const std::string& n) const
	{
		auto it = mNamed.find(n);
		return it == mNamed.end() ? PR_INVALID_ID : it->second;
	}
	std::shared_ptr<T> getSafe(uint32 id) const { return id < mObjects.size() ? mObjects[id] : nullptr; }
	const std::vector<std::shared_ptr<T>>& getAll() const { return mObjects; }
	size_t size() const { return mObjects.size(); }

private:
	std::vector<std::shared_ptr<T>> mObjects;
	std::map<std::string, uint32> mNamed;
};
struct SceneDatabase { // reference src/core/scene/SceneDatabase.h:19-29
	AbstractDatabase<IEntity> Entities;
	AbstractDatabase<IMaterial> Materials;
	AbstractDatabase<IEmission> Emissions;
	AbstractDatabase<IInfiniteLight> InfiniteLights;
	AbstractDatabase<INode> Nodes;
};

struct RenderSettings { // reference src/core/renderer/RenderSettings.cpp:11-33
	uint64 seed				   = 42;
	uint32 maxParallelRays	   = 10000;
	uint32 sampleCountOverride = 0;
	float timeScale			   = 1;
	bool useAdaptiveTiling	   = true;
	bool sortHits			   = false;
	bool progressive		   = false;
	float spectralStart		   = PR_CIE_WAVELENGTH_START;
	float spectralEnd		   = PR_CIE_WAVELENGTH_END;
	bool spectralMono		   = false;
	bool spectralHero		   = true;
	uint32 filmWidth = 1920, filmHeight = 1080;
	float cropMinX = 0, cropMaxX = 1, cropMinY = 0, cropMaxY = 1;
	std::shared_ptr<ISamplerFactory> aaSamplerFactory, lensSamplerFactory, timeSamplerFactory, spectralSamplerFactory;
	std::shared_ptr<IFilterFactory> pixelFilterFactory;
	std::shared_ptr<IIntegratorFactory> integratorFactory;
	std::map<std::string, std::shared_ptr<ISpectralMapperFactory>> spectralMapperFactories;
	uint32 maxSampleCount() const; // RenderSettings.cpp:76-88
	// crop window in pixels (reference RenderSettings.h cropPixelOffset/cropWidth/..)
	uint32 cropWidth() const { return (uint32)((cropMaxX - cropMinX) * filmWidth); }
	uint32 cropHeight() const { return (uint32)((cropMaxY - cropMinY) * filmHeight); }
	uint32 cropOffsetX() const { return (uint32)(cropMinX * filmWidth); }
	uint32 cropOffsetY() const { return (uint32)(cropMinY * filmHeight); }
};

// ------------------------------------------------------------------ light path expressions (lpe.cpp)
// reference src/core/path/LightPathExpression.h; dense DFA over the 15 (ScatteringType, ScatteringEvent) symbols
constexpr uint8_t LPE_REJECT = 0xFF;
struct LPEAutomaton {
	bool valid		  = false;
	uint32 stateCount = 0;	   // state 0 is the start state
	std::vector<uint8_t> next; // [state * 15 + type * 3 + event] -> state or LPE_REJECT
	std::vector<uint8_t> final;
	bool match(const std::vector<std::pair<int, int>>& tokens) const; // (type, event) pairs, LightPathToken.h:6-20
};
LPEAutomaton compileLPE(const std::string& expression);

// ------------------------------------------------------------------ output specification + image writer (image_io.cpp)
enum class ToneColorMode { SRGB, XYZ, XYZNorm, Luminance }; // reference src/core/spectral/ToneMapper.h
enum OutputVariable {
	OV_Unsupported = -1,
	OV_Output	   = 0,
	OV_Position,
	OV_Normal,
	OV_UVW,
	OV_Depth,
	OV_EntityID,
	OV_SampleCount,
	OV_Feedback,
	OV_OnlineMean,
	OV_OnlineVariance,
	OV_NormalG,
	OV_Tangent,
	OV_Bitangent,
	OV_View,
	OV_MaterialID,
	OV_EmissionID,
	OV_DisplaceID
};
struct OutputChannel { // reference IM_ChannelSetting{Spec,3D,1D,Counter}, src/loader/output/io/ImageWriter.h
	enum Kind { Spectral, ThreeD, OneD, Counter } kind = Spectral;
	int variable	  = OV_Output;
	ToneColorMode tcm = ToneColorMode::SRGB;
	std::string name; // empty for the plain colour channel ("R", "G", "B")
	std::string lpe;  // light path expression restricting the channel ("" = none)
	int lpeIndex = -1; // spectral channels: index into the scene's LPE list (OutputSpecification::lpeExpressions)
};
struct OutputFile {
	std::string name;
	std::vector<OutputChannel> channels;
};
struct FilmView { // what prb_film_download / prb_film_aov return for one context
	uint32 width = 0, height = 0;		  // view size
	uint32 offsetX = 0, offsetY = 0;	  // view offset inside the film
	uint32 fullWidth = 0, fullHeight = 0; // film size
	const float* xyz		  = nullptr;  // 3 per pixel
	const uint32* sampleCount = nullptr;  // 1 per pixel
	const uint32* feedback	  = nullptr;  // 1 per pixel: OR of PRB_FEEDBACK_* bits; may be null
	const float* onlineMean		= nullptr; // 3 per pixel (AOV_OnlineMean); may be null
	const float* onlineVariance = nullptr; // 3 per pixel (AOV_OnlineVariance); may be null
	const float* aov		  = nullptr;  // 10 per pixel (N, P, u, v, depth, entity id), sums over the samples; may be null
	const float* aovExt		  = nullptr;  // PRB_AOV_EXT per pixel (tangent, bitangent, view, material id, emission id), sums; may be null
	std::vector<const float*> lpe;		  // per light path expression of the scene: 3 per pixel (XYZ), may be empty / null entries
};
class OutputSpecification { // reference src/loader/output/io/OutputSpecification.h
public:
	void parse(const DL::DataGroup& entry);
	const std::vector<OutputFile>& files() const { return mFiles; }
	// does any channel ask for the online mean / variance AOVs (FrameOutputData::hasVarianceEstimator)?
	bool wantsVariance() const
	{
		for (const OutputFile& f : mFiles)
			for (const OutputChannel& c : f.channels)
				if (c.variable == OV_OnlineMean || c.variable == OV_OnlineVariance)
					return true;
		return false;
	}
	// does any channel ask for an AOV of prb_film_download_aov_ext (tangent, bitangent, view, material / emission id)?
	bool wantsExtendedAOVs() const
	{
		for (const OutputFile& f : mFiles)
			for (const OutputChannel& c : f.channels)
				if (c.variable == OV_Tangent || c.variable == OV_Bitangent || c.variable == OV_View || c.variable == OV_MaterialID || c.variable == OV_EmissionID)
					return true;
		return false;
	}
	// the distinct light path expressions of the spectral channels, in registration order (prb_scene_desc::lpe)
	const std::vector<std::string>& lpeExpressions() const { return mLPEs; }
	// writes <workingDir>/results[_<contextIndex>]/<name>.exr for every (output ...) block; returns the number written
	int save(const std::string& workingDir, const FilmView& film, uint32 contextIndex = 0) const;

private:
	std::vector<OutputFile> mFiles;
	std::vector<std::string> mLPEs;
};
bool saveImage(const std::string& path, const OutputFile& file, const FilmView& film);
// image files for texture nodes (image_read.cpp): EXR scanline (half / float; none, ZIPS, ZIP), PFM, binary PPM / PGM
struct ImageData {
	uint32 width = 0, height = 0, channels = 0; // 1 or 3 channels, rows top to bottom
	bool linear = true;							// false: sRGB encoded (integer formats)
	std::vector<float> data;
};
bool loadImage(const std::string& path, ImageData& img);
bool writeEXR(const std::string& path, const std::vector<std::string>& channelNames, const std::vector<const float*>& planes, uint32 width, uint32 height,
			  int32_t offX, int32_t offY, uint32 fullWidth, uint32 fullHeight);

class Environment { // reference src/loader/Environment.h:45-134
public:
	explicit Environment(const std::string& pluginPath = "");
	RenderSettings& renderSettings() { return mRenderSettings; }
	const RenderSettings& renderSettings() const { return mRenderSettings; }
	SceneDatabase* sceneDatabase() { return &mDatabase; }
	const SceneDatabase* sceneDatabase() const { return &mDatabase; }
	const std::shared_ptr<SpectralUpsampler>& defaultSpectralUpsampler() const { return mUpsampler; }
	OutputSpecification& outputSpecification() { return mOutputSpecification; }
	const OutputSpecification& outputSpecification() const { return mOutputSpecification; }

private:
	// Declared FIRST so that it is destroyed LAST: the factories below and every object they created (materials, nodes ...
	// held by the scene database) may live in an external plugin library, which ~PluginManager unloads (the reference keeps
	// the same order: "library unloaded after plugin reset", loader/plugin/PluginManager.h:38-50).
	PluginManager mPluginManager;

public:
	AbstractManager<ICameraPlugin> cameraManager;
	AbstractManager<IEmissionPlugin> emissionManager;
	AbstractManager<IEntityPlugin> entityManager;
	AbstractManager<IFilterPlugin> filterManager;
	AbstractManager<IInfiniteLightPlugin> infiniteLightManager;
	AbstractManager<IIntegratorPlugin> integratorManager;
	AbstractManager<IMaterialPlugin> materialManager;
	AbstractManager<INodePlugin> nodeManager;
	AbstractManager<ISamplerPlugin> samplerManager;
	AbstractManager<ISpectralMapperPlugin> spectralMapperManager;

	std::map<std::string, std::shared_ptr<MeshBase>> meshes;
	std::map<std::string, std::shared_ptr<INode>> namedNodes;
	std::shared_ptr<ICamera> activeCamera;
	std::string sceneName;

	// reference SamplerManager/FilterManager/SpectralMapperManager::createDefaultsIfNecessary + default integrator
	bool createDefaultsIfNecessary();

private:
	RenderSettings mRenderSettings;
	SceneDatabase mDatabase;
	std::shared_ptr<SpectralUpsampler> mUpsampler;
	OutputSpecification mOutputSpecification;
};

class SceneLoadContext { // reference src/loader/SceneLoadContext.h / .cpp:196-326
public:
	SceneLoadContext(Environment* env, const std::string& file = "")
		: mEnv(env)
	{
		if (!file.empty())
			mFileStack.push_back(file);
	}
	Environment* environment() const { return mEnv; }
	ParameterGroup& parameters() { return mParameters; }
	const ParameterGroup& parameters() const { return mParameters; }
	Transformf& transform() { return mTransform; }
	const Transformf& transform() const { return mTransform; }
	std::string currentFile() const { return mFileStack.empty() ? "" : mFileStack.back(); }
	void pushFile(const std::string& f) { mFileStack.push_back(f); }
	void popFile() { mFileStack.pop_back(); }
	std::string setupParametricPath(const std::string& p) const; // relative to the including file

	std::shared_ptr<INode> getRawNode(uint32 id) const { return mEnv->sceneDatabase()->Nodes.getSafe(id); }
	std::shared_ptr<INode> getRawNode(const std::string& name) const;
	std::shared_ptr<FloatSpectralNode> lookupSpectralNode(const Parameter& p, float def = 1) const;
	std::shared_ptr<FloatSpectralNode> lookupSpectralNode(const std::string& name, float def = 1) const { return lookupSpectralNode(mParameters.getParameter(name), def); }
	std::shared_ptr<FloatSpectralNode> lookupSpectralNode(const std::initializer_list<std::string>& names, float def = 1) const;
	std::shared_ptr<FloatScalarNode> lookupScalarNode(const Parameter& p, float def = 1) const;
	std::shared_ptr<FloatScalarNode> lookupScalarNode(const std::string& name, float def = 1) const { return lookupScalarNode(mParameters.getParameter(name), def); }
	std::shared_ptr<FloatScalarNode> lookupScalarNode(const std::initializer_list<std::string>& names, float def = 1) const;
	uint32 lookupMaterialID(const Parameter& p) const;
	std::vector<uint32> lookupMaterialIDArray(const Parameter& p) const;
	uint32 lookupEmissionID(const Parameter& p) const;
	bool hasMesh(const std::string& n) const { return mEnv->meshes.count(n) > 0; }
	std::shared_ptr<MeshBase> getMesh(const std::string& n) const { return mEnv->meshes.at(n); }
	std::shared_ptr<IMaterial> loadMaterial(const std::string& type, const ParameterGroup& params) const;
	std::shared_ptr<ISamplerFactory> loadSamplerFactory(const std::string& type, const ParameterGroup& params) const;

private:
	Environment* mEnv;
	ParameterGroup mParameters;
	Transformf mTransform;
	std::vector<std::string> mFileStack;
};

struct SceneLoadOptions { // reference SceneLoader::LoadOptions
	std::string PluginPath;
	bool Progressive = false;
};
class SceneLoader { // reference src/loader/SceneLoader.cpp:44-1041
public:
	using LoadOptions = SceneLoadOptions;
	static std::shared_ptr<Environment> loadFromFile(const std::string& path, const LoadOptions& opts = LoadOptions());
	static std::shared_ptr<Environment> loadFromString(const std::string& source, const std::string& virtualPath = "", const LoadOptions& opts = LoadOptions());

private:
	static std::shared_ptr<Environment> createEnvironment(const std::vector<DL::DataGroup>& groups, const LoadOptions& opts, const std::string& path);
	static void setupEnvironment(const std::vector<DL::DataGroup>& groups, SceneLoadContext& ctx);
	static void addSampler(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addFilter(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addIntegrator(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addSpectralMapper(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addEntity(const DL::DataGroup& g, const ITransformable* parent, SceneLoadContext& ctx);
	static void addCamera(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addLight(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addEmission(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addMaterial(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addNode(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addTexture(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addMesh(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addInclude(const DL::DataGroup& g, SceneLoadContext& ctx);
	static void addSubGraph(const DL::DataGroup& g, SceneLoadContext& ctx); // (embed :loader 'obj' ...)
	static uint32 addNodeInline(const DL::DataGroup& g, SceneLoadContext& ctx);
	static Transformf extractTransform(const DL::DataGroup& g);
	static ParameterGroup populateObjectParameters(const DL::DataGroup& g, SceneLoadContext& ctx);
	static Parameter unpackShadingNetwork(const DL::DataGroup& g, SceneLoadContext& ctx);
};

// ------------------------------------------------------------------ lights
class Light { // reference src/core/light/Light.h
public:
	uint32 id				 = 0;
	IEntity* entity			 = nullptr; // area
	IEmission* emission		 = nullptr;
	IInfiniteLight* infLight = nullptr;
	float relContribution	 = 0;
	bool isInfinite() const { return infLight != nullptr; }
	SpectralBlob averagePower(const SpectralBlob& wvl) const { return isInfinite() ? infLight->power(wvl) : emission->power(wvl); }
	SpectralRange spectralRange() const { return isInfinite() ? infLight->spectralRange() : emission->spectralRange(); }
};
class LightSampler { // reference src/core/light/LightSampler.cpp:11-132
public:
	LightSampler(const SceneDatabase& db, float sceneBoundingSphereRadius, const SpectralRange& cameraRange);
	const std::vector<Light>& lights() const { return mLights; }
	const Distribution1D& selector() const { return mSelector; }
	SpectralRange lightSpectralRange() const { return mLightSpectralRange; }
	float infLightSelectionProbability() const { return mInfLightSelectionProbability; }
	float emissiveSurfaceArea() const { return mEmissiveSurfaceArea; }
	float emissivePower() const { return mEmissivePower; }

private:
	std::vector<Light> mLights;
	Distribution1D mSelector;
	float mInfLightSelectionProbability = 0, mEmissiveSurfaceArea = 0, mEmissiveSurfacePower = 0, mEmissivePower = 0;
	SpectralRange mLightSpectralRange;
};

// ------------------------------------------------------------------ BVH builder (host; replaces rtcCommitScene, Scene.cpp:99-101)
struct BVHBuildInput {
	std::vector<BoundingBox> boxes; // one per primitive
};
struct BVH8 {
	std::vector<prb_bvh8_node> nodes; // root at index 0
	std::vector<uint32> primOrder;	  // leaf-ordered primitive indices (prim_base/offset index into this)
	BoundingBox bounds;
};
BVH8 buildBVH8(const BVHBuildInput& in, int maxLeafPrims);

// ------------------------------------------------------------------ scene compiler
// Flattens an Environment into the POD descriptor (owning all arrays).
class CompiledScene {
public:
	prb_scene_desc desc{};
	prb_integrator integrator{ PRB_INTEGRATOR_DIRECT, 0 }; // the scene's (integrator ...) block, for prb_set_integrator
	std::vector<prb_node> nodes;
	std::vector<prb_material> materials;
	std::vector<prb_emission> emissions;
	std::vector<prb_entity> entities;
	std::vector<uint32> entityMaterials;
	std::vector<prb_mesh> meshes;
	std::vector<float> vertices, normals, uvs;
	std::vector<uint32> faceIndices, faceSlots;
	std::vector<prb_light> lights;
	std::vector<float> lightCDF;
	std::vector<prb_bvh8_node> bvhNodes;
	std::vector<prb_bvh_tri> bvhTris;
	std::vector<uint32> tlasRefs;
	std::vector<float> pool;
	std::vector<uint8_t> lpeTables;
	BoundingBox sceneBounds;
	float sceneRadius = 0;
	double bvhBuildSeconds = 0;
	void finalize(); // point desc at the vectors
};
class SceneCompiler {
public:
	explicit SceneCompiler(Environment* env)
		: mEnv(env)
	{
	}
	std::shared_ptr<CompiledScene> compile();
	// used by IEntity::describe
	uint32 registerMesh(const std::shared_ptr<MeshBase>& mesh);
	uint32 registerEntityMaterials(const std::vector<uint32>& ids);
	CompiledScene& scene() { return *mScene; }

private:
	Environment* mEnv;
	std::shared_ptr<CompiledScene> mScene;
	std::map<const MeshBase*, uint32> mMeshIDs;
};
// synthetic triangle soup (SURVEY 8(d) C5): one identity-transform mesh of n triangles + pinhole camera
std::shared_ptr<CompiledScene> makeSoupScene(uint32 triangles, uint64 seed, uint32 filmW, uint32 filmH);

// reference RenderRandomMap.cpp:11-28 (warm-up by jump-ahead + libstdc++ permutation)
std::vector<uint64> buildRenderRandomMap(uint64 seed, uint32 width, uint32 height, uint32 rngDelta);

// ------------------------------------------------------------------ render driver
struct RenderTile { // reference src/core/renderer/RenderTile.h (start/end only)
	uint32 sx, sy, ex, ey;
};
// reference RenderTileMap::init (RenderTileMap.cpp:26-122): rtx x rty tiles over the view, Z-order
std::vector<RenderTile> buildTileMap(uint32 viewX, uint32 viewY, uint32 viewW, uint32 viewH, uint32 rtx, uint32 rty);

class RenderTileSession { // reference src/core/renderer/RenderTileSession.h (what the device path needs)
public:
	RenderTileSession(RenderContext* ctx, const RenderTile* tile, uint32 iteration)
		: mContext(ctx)
		, mTile(tile)
		, mIteration(iteration)
	{
	}
	RenderContext* context() const { return mContext; }
	const RenderTile* tile() const { return mTile; }
	uint32 iteration() const { return mIteration; }

private:
	RenderContext* mContext;
	const RenderTile* mTile;
	uint32 mIteration;
};

class RenderContext { // reference src/core/renderer/RenderContext.cpp:65-139,234-296
public:
	RenderContext(const std::shared_ptr<Environment>& env, int device, uint32 rank = 0, uint32 worldSize = 1);
	~RenderContext();
	bool valid() const { return mCtx != nullptr; }
	// runs all iterations of all tiles this rank owns (interleaved tile_id % worldSize == rank)
	bool start(uint32 rtx, uint32 rty, uint32 iterations = 0);
	void waitForFinish();
	const std::shared_ptr<CompiledScene>& compiledScene() const { return mScene; }
	prb_ctx* deviceContext() const { return mCtx; }
	std::vector<float> filmXYZ();
	// writes <workingDir>/results[_<rank>]/<name>.exr for every (output ...) block of the scene; returns the number of files
	int saveOutputs(const std::string& workingDir);
	prb_stats statistics() const;
	const RenderSettings& settings() const { return mEnv->renderSettings(); }
	const std::vector<RenderTile>& ownedTiles() const { return mOwnedTiles; }
	// One process per GPU: joins the NCCL communicator of the job (id from prb_comm_unique_id of rank 0, shipped out of
	// band); start() then ends with prb_film_reduce_comm, after which rank 0 holds the combined film.
	bool joinCommunicator(const uint8_t id[PRB_COMM_UNIQUE_ID_BYTES]);
	// One process driving several GPUs: combines the films of contexts[1..] into contexts[0] (prb_film_reduce).  The
	// counterpart of the reference client merging its image-tile contexts (RenderFactory.cpp:16-42, client/main.cpp:172-173).
	static bool combineFilms(const std::vector<RenderContext*>& contexts);

private:
	std::shared_ptr<Environment> mEnv;
	std::shared_ptr<CompiledScene> mScene;
	std::shared_ptr<IIntegrator> mIntegrator;
	prb_ctx* mCtx = nullptr;
	uint32 mRank, mWorldSize;
	bool mHasCommunicator = false;
	std::vector<RenderTile> mOwnedTiles;
};
} // namespace PR
