// Environment, plugin manager, scene-load context and the .prc scene loader
// (reference src/loader/{Environment,SceneLoadContext,SceneLoader}.cpp, plugin/PluginManager.cpp).
#include "prh.h"

#include <dirent.h>
#include <sys/stat.h>

#include <dlfcn.h>
#include <fstream>
#include <map>
#include <sstream>
#include <tuple>

namespace PR {
void registerNodePlugins(std::vector<std::shared_ptr<IPlugin>>& out);
void registerMaterialPlugins(std::vector<std::shared_ptr<IPlugin>>& out);
void registerScenePlugins(std::vector<std::shared_ptr<IPlugin>>& out);
std::vector<std::shared_ptr<IPlugin>> createSkySunPlugins(); // skysun.cpp
void registerEmbeddedPlugins(std::vector<std::shared_ptr<IPlugin>>& out)
{
	registerNodePlugins(out);
	registerMaterialPlugins(out);
	registerScenePlugins(out);
	for (const auto& p : createSkySunPlugins())
		out.push_back(p);
}

// ------------------------------------------------------------------ PluginManager
PluginManager::PluginManager(const std::string& pluginPath)
{
	loadEmbeddedPlugins();
	// external plugins (PluginManager::initPlugins / loadFromDirectory, PluginManager.cpp:14-66): every entry of the ':' separated
	// plugin path and of the environment variable PR_PLUGIN_PATH is a DIRECTORY searched for (lib)?pr_pl_<name>.so, or -- an
	// extension -- one such file given explicitly; each object must export `_pr_exports` (Plugin.h:52-66).
	std::string paths = pluginPath;
	if (const char* e = std::getenv("PR_PLUGIN_PATH")) {
		if (!paths.empty())
			paths += ":";
		paths += e;
	}
	size_t pos = 0;
	while (pos < paths.size()) {
		size_t end = paths.find(':', pos);
		if (end == std::string::npos)
			end = paths.size();
		const std::string f = paths.substr(pos, end - pos);
		pos					= end + 1;
		if (f.empty())
			continue;
		struct stat sb;
		if (stat(f.c_str(), &sb) != 0)
			continue;
		if (S_ISDIR(sb.st_mode)) {
			std::vector<std::string> found;
			if (DIR* dir = opendir(f.c_str())) {
				while (const dirent* de = readdir(dir)) {
					std::string n = de->d_name;
					if (n.size() <= 3 || n.substr(n.size() - 3) != ".so")
						continue;
					std::string stem = n.substr(0, n.size() - 3);
					if (stem.rfind("lib", 0) == 0)
						stem = stem.substr(3);
					if (stem.rfind("pr_pl_", 0) != 0 || stem.size() <= 6)
						continue;
					if (stem.size() > 2 && stem.substr(stem.size() - 2) == "_d") // debug builds are ignored, PluginManager.cpp:52-56
						continue;
					found.push_back(f + "/" + n);
				}
				closedir(dir);
			}
			std::sort(found.begin(), found.end());
			for (const std::string& so : found)
				tryLoad(so);
		} else if (f.size() > 3 && f.substr(f.size() - 3) == ".so") {
			tryLoad(f);
		}
	}
}
PluginManager::~PluginManager()
{
	mPlugins.clear();
	for (void* l : mLibraries)
		dlclose(l);
}
void PluginManager::loadEmbeddedPlugins() { registerEmbeddedPlugins(mPlugins); }
bool PluginManager::tryLoad(const std::string& path)
{
	void* lib = dlopen(path.c_str(), RTLD_NOW | RTLD_LOCAL);
	if (!lib) {
		PR_LOG(L_ERROR) << "Could not load plugin " << path << ": " << dlerror() << std::endl;
		return false;
	}
	auto* ptr = reinterpret_cast<PluginInterface*>(dlsym(lib, "_pr_exports"));
	if (!ptr) {
		PR_LOG(L_ERROR) << "Could not get file interface for " << path << std::endl;
		dlclose(lib);
		return false;
	}
	if (ptr->APIVersion < PR_PLUGIN_API_VERSION) {
		PR_LOG(L_ERROR) << "Plugin " << path << " has old API version " << ptr->APIVersion << ", expected " << PR_PLUGIN_API_VERSION << std::endl;
		dlclose(lib);
		return false;
	}
	if (ptr->APIVersion > PR_PLUGIN_API_VERSION) {
		PR_LOG(L_ERROR) << "Plugin " << path << " has newer API version " << ptr->APIVersion << ", expected " << PR_PLUGIN_API_VERSION << std::endl;
		dlclose(lib);
		return false;
	}
	IPlugin* p = ptr->InitFunction();
	if (!p) {
		PR_LOG(L_ERROR) << "Could not initialize plugin " << path << std::endl;
		dlclose(lib);
		return false;
	}
	mLibraries.push_back(lib);
	mPlugins.emplace_back(p);
	return true;
}

// ------------------------------------------------------------------ Environment
std::string dataDirectory()
{
	if (const char* e = std::getenv("PRB200_DATA_DIR"))
		return e;
	Dl_info info;
	if (dladdr(reinterpret_cast<void*>(&dataDirectory), &info) && info.dli_fname) {
		std::string p = info.dli_fname; // .../pearray_b200/libprb200_host.so
		size_t s	  = p.find_last_of('/');
		if (s != std::string::npos)
			return p.substr(0, s) + "/data";
	}
	return "pearray_b200/data";
}

Environment::Environment(const std::string& pluginPath)
	: mPluginManager(pluginPath)
{
	mUpsampler = std::make_shared<SpectralUpsampler>(dataDirectory() + "/rgb2spec_srgb.bin");
	for (const auto& p : mPluginManager.plugins()) { // routing by IPlugin::type(), Environment.cpp:203-241
		switch (p->type()) {
		case PluginType::Camera: cameraManager.addFactory(std::dynamic_pointer_cast<ICameraPlugin>(p)); break;
		case PluginType::Emission: emissionManager.addFactory(std::dynamic_pointer_cast<IEmissionPlugin>(p)); break;
		case PluginType::Entity: entityManager.addFactory(std::dynamic_pointer_cast<IEntityPlugin>(p)); break;
		case PluginType::Filter: filterManager.addFactory(std::dynamic_pointer_cast<IFilterPlugin>(p)); break;
		case PluginType::InfiniteLight: infiniteLightManager.addFactory(std::dynamic_pointer_cast<IInfiniteLightPlugin>(p)); break;
		case PluginType::Integrator: integratorManager.addFactory(std::dynamic_pointer_cast<IIntegratorPlugin>(p)); break;
		case PluginType::Material: materialManager.addFactory(std::dynamic_pointer_cast<IMaterialPlugin>(p)); break;
		case PluginType::Node: nodeManager.addFactory(std::dynamic_pointer_cast<INodePlugin>(p)); break;
		case PluginType::Sampler: samplerManager.addFactory(std::dynamic_pointer_cast<ISamplerPlugin>(p)); break;
		case PluginType::SpectralMapper: spectralMapperManager.addFactory(std::dynamic_pointer_cast<ISpectralMapperPlugin>(p)); break;
		}
	}
	// built-in named colour nodes, Environment.cpp:83-102
	struct C {
		const char* n;
		float r, g, b;
	};
	static const C colors[] = { { "black", 0, 0, 0 }, { "white", 1, 1, 1 }, { "red", 1, 0, 0 }, { "green", 0, 1, 0 }, { "blue", 0, 0, 1 },
								{ "magenta", 1, 0, 1 }, { "yellow", 1, 1, 0 }, { "cyan", 0, 1, 1 }, { "gray", 0.5f, 0.5f, 0.5f },
								{ "lightGray", 0.666f, 0.666f, 0.666f }, { "darkGray", 0.333f, 0.333f, 0.333f } };
	auto fac = nodeManager.getFactory("refl");
	for (const C& c : colors) {
		SceneLoadContext ctx(this);
		ctx.parameters().addParameter(Parameter::fromNumber(c.r));
		ctx.parameters().addParameter(Parameter::fromNumber(c.g));
		ctx.parameters().addParameter(Parameter::fromNumber(c.b));
		if (fac)
			namedNodes[c.n] = fac->create("refl", ctx);
	}
}

bool Environment::createDefaultsIfNecessary()
{
	auto& s = mRenderSettings;
	auto mkSampler = [&](const char* type, int sc) -> std::shared_ptr<ISamplerFactory> {
		auto fac = samplerManager.getFactory(type);
		if (!fac)
			return nullptr;
		SceneLoadContext ctx(this);
		ctx.parameters().addParameter("sample_count", Parameter::fromInt(sc));
		return fac->create(type, ctx);
	};
	if (!s.aaSamplerFactory) { // SamplerManager.cpp:14-72
		PR_LOG(L_WARNING) << "No AA sampler selected. Using " << (s.progressive ? "multi jittered" : "sobol") << " sampler with sample count 128" << std::endl;
		s.aaSamplerFactory = mkSampler(s.progressive ? "mjitt" : "sobol", 128);
	}
	if (!s.lensSamplerFactory)
		s.lensSamplerFactory = mkSampler("random", 1);
	if (!s.timeSamplerFactory)
		s.timeSamplerFactory = mkSampler("random", 1);
	if (!s.spectralSamplerFactory)
		s.spectralSamplerFactory = mkSampler("random", 1);
	if (!s.pixelFilterFactory) { // FilterManager.cpp: mitchell radius 1
		auto fac = filterManager.getFactory("mitchell");
		SceneLoadContext ctx(this);
		ctx.parameters().addParameter("radius", Parameter::fromInt(1));
		if (fac)
			s.pixelFilterFactory = fac->create("mitchell", ctx);
	}
	if (!s.spectralMapperFactories.count("pixel")) { // SpectralMapperManager.cpp:30
		auto fac = spectralMapperManager.getFactory("spd");
		SceneLoadContext ctx(this);
		if (fac)
			s.spectralMapperFactories["pixel"] = fac->create("spd", ctx);
	}
	if (!s.spectralMapperFactories.count("light"))
		s.spectralMapperFactories["light"] = s.spectralMapperFactories["pixel"];
	if (!s.integratorFactory) { // IntegratorManager default: 'direct'
		PR_LOG(L_WARNING) << "No integrator selected. Using direct integrator" << std::endl;
		auto fac = integratorManager.getFactory("direct");
		SceneLoadContext ctx(this);
		if (fac)
			s.integratorFactory = fac->create("direct", ctx);
	}
	return s.aaSamplerFactory && s.lensSamplerFactory && s.timeSamplerFactory && s.spectralSamplerFactory && s.pixelFilterFactory
		   && s.spectralMapperFactories["pixel"] && s.integratorFactory;
}

// ------------------------------------------------------------------ SceneLoadContext
std::string SceneLoadContext::setupParametricPath(const std::string& p) const
{
	if (p.empty() || p[0] == '/')
		return p;
	const std::string cur = currentFile();
	const size_t s		  = cur.find_last_of('/');
	if (s == std::string::npos)
		return p;
	return cur.substr(0, s + 1) + p;
}
std::shared_ptr<INode> SceneLoadContext::getRawNode(const std::string& name) const
{
	auto it = mEnv->namedNodes.find(name);
	return it == mEnv->namedNodes.end() ? nullptr : it->second;
}
std::shared_ptr<FloatSpectralNode> SceneLoadContext::lookupSpectralNode(const Parameter& p, float def) const
{ // SceneLoadContext.cpp:196-230
	switch (p.type()) {
	default: return makeConstSpectralNode(def);
	case ParameterType::Int:
	case ParameterType::UInt:
	case ParameterType::Number:
		if (p.isArray())
			return makeConstSpectralNode(def);
		return makeConstSpectralNode(p.getNumber(0.0f));
	case ParameterType::Reference: {
		const auto node = getRawNode(p.getReference());
		if (node && node->type() == NodeType::FloatSpectral)
			return std::static_pointer_cast<FloatSpectralNode>(node);
		if (node && node->type() == NodeType::FloatScalar) // SplatSpectralNode of a constant
			return makeConstSpectralNode(std::static_pointer_cast<FloatScalarNode>(node)->eval(ShadingContext()));
		return makeConstSpectralNode(def);
	}
	case ParameterType::String: {
		const auto node = getRawNode(p.getString(""));
		if (node && node->type() == NodeType::FloatSpectral)
			return std::static_pointer_cast<FloatSpectralNode>(node);
		return makeConstSpectralNode(def);
	}
	}
}
std::shared_ptr<FloatSpectralNode> SceneLoadContext::lookupSpectralNode(const std::initializer_list<std::string>& names, float def) const
{
	for (const auto& n : names)
		if (mParameters.hasParameter(n))
			return lookupSpectralNode(mParameters.getParameter(n), def);
	return lookupSpectralNode(mParameters.getParameter(*names.begin()), def);
}
std::shared_ptr<FloatScalarNode> SceneLoadContext::lookupScalarNode(const Parameter& p, float def) const
{ // SceneLoadContext.cpp:232-262
	switch (p.type()) {
	default: return makeConstScalarNode(def);
	case ParameterType::Int:
	case ParameterType::UInt:
	case ParameterType::Number:
		if (p.isArray())
			return makeConstScalarNode(def);
		return makeConstScalarNode(p.getNumber(def));
	case ParameterType::Reference: {
		const auto node = getRawNode(p.getReference());
		if (node && node->type() == NodeType::FloatScalar)
			return std::static_pointer_cast<FloatScalarNode>(node);
		return makeConstScalarNode(def);
	}
	case ParameterType::String: {
		const auto node = getRawNode(p.getString(""));
		if (node && node->type() == NodeType::FloatScalar)
			return std::static_pointer_cast<FloatScalarNode>(node);
		return makeConstScalarNode(def);
	}
	}
}
std::shared_ptr<FloatScalarNode> SceneLoadContext::lookupScalarNode(const std::initializer_list<std::string>& names, float def) const
{
	for (const auto& n : names)
		if (mParameters.hasParameter(n))
			return lookupScalarNode(mParameters.getParameter(n), def);
	return lookupScalarNode(mParameters.getParameter(*names.begin()), def);
}
uint32 SceneLoadContext::lookupMaterialID(const Parameter& p) const
{
	if (p.type() != ParameterType::String)
		return PR_INVALID_ID;
	const std::string name = p.getString("");
	if (!mEnv->sceneDatabase()->Materials.has(name)) {
		PR_LOG(L_ERROR) << "Could not find material " << name << std::endl;
		return PR_INVALID_ID;
	}
	return mEnv->sceneDatabase()->Materials.getID(name);
}
std::vector<uint32> SceneLoadContext::lookupMaterialIDArray(const Parameter& p) const
{
	std::vector<uint32> r;
	if (p.type() != ParameterType::String)
		return r;
	const size_t n = p.isArray() ? p.arraySize() : 1;
	for (size_t i = 0; i < n; ++i) {
		const std::string name = p.getString(i, "");
		if (!mEnv->sceneDatabase()->Materials.has(name)) {
			PR_LOG(L_ERROR) << "Could not find material " << name << std::endl;
			r.push_back(PR_INVALID_ID);
		} else {
			r.push_back(mEnv->sceneDatabase()->Materials.getID(name));
		}
	}
	return r;
}
uint32 SceneLoadContext::lookupEmissionID(const Parameter& p) const
{
	if (p.type() != ParameterType::String)
		return PR_INVALID_ID;
	const std::string name = p.getString("");
	if (name.empty())
		return PR_INVALID_ID;
	if (!mEnv->sceneDatabase()->Emissions.has(name)) {
		PR_LOG(L_ERROR) << "Could not find emission " << name << std::endl;
		return PR_INVALID_ID;
	}
	return mEnv->sceneDatabase()->Emissions.getID(name);
}
std::shared_ptr<IMaterial> SceneLoadContext::loadMaterial(const std::string& type, const ParameterGroup& params) const
{
	auto fac = mEnv->materialManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "Unknown material type " << type << std::endl;
		return nullptr;
	}
	SceneLoadContext ctx = *this;
	ctx.parameters()	 = params;
	return fac->create(type, ctx);
}
std::shared_ptr<ISamplerFactory> SceneLoadContext::loadSamplerFactory(const std::string& type, const ParameterGroup& params) const
{
	auto fac = mEnv->samplerManager.getFactory(type);
	if (!fac)
		return nullptr;
	SceneLoadContext ctx = *this;
	ctx.parameters()	 = params;
	return fac->create(type, ctx);
}

// ------------------------------------------------------------------ SceneLoader
static std::string lower(std::string s)
{
	std::transform(s.begin(), s.end(), s.begin(), [](char c) { return (char)std::tolower(c); });
	return s;
}

std::shared_ptr<Environment> SceneLoader::loadFromFile(const std::string& path, const LoadOptions& opts)
{
	try {
		return createEnvironment(DL::parseFile(path), opts, path);
	} catch (const std::exception& e) {
		PR_LOG(L_ERROR) << e.what() << std::endl;
		return nullptr;
	}
}
std::shared_ptr<Environment> SceneLoader::loadFromString(const std::string& source, const std::string& virtualPath, const LoadOptions& opts)
{
	try {
		return createEnvironment(DL::parseString(source), opts, virtualPath);
	} catch (const std::exception& e) {
		PR_LOG(L_ERROR) << e.what() << std::endl;
		return nullptr;
	}
}

std::shared_ptr<Environment> SceneLoader::createEnvironment(const std::vector<DL::DataGroup>& groups, const LoadOptions& opts, const std::string& path)
{ // SceneLoader.cpp:73-151
	if (groups.empty()) {
		PR_LOG(L_ERROR) << "DataLisp file does not contain valid entries" << std::endl;
		return nullptr;
	}
	const DL::DataGroup& top = groups.front();
	if (top.id() != "scene") {
		PR_LOG(L_ERROR) << "DataLisp file does not contain valid top entry" << std::endl;
		return nullptr;
	}
	auto env					 = std::make_shared<Environment>(opts.PluginPath);
	RenderSettings& rs			 = env->renderSettings();
	rs.progressive				 = opts.Progressive;
	const DL::Data nameD		 = top.getFromKey("name");
	const DL::Data renderWidthD	 = top.getFromKey("render_width");
	const DL::Data renderHeightD = top.getFromKey("render_height");
	const DL::Data cropD		 = top.getFromKey("crop");
	const DL::Data spectralDomainD = top.getFromKey("spectral_domain");
	const DL::Data spectralHeroD   = top.getFromKey("spectral_hero");
	if (nameD.type() == DL::DT_String)
		env->sceneName = nameD.getString();
	if (renderWidthD.type() == DL::DT_Integer)
		rs.filmWidth = (uint32)renderWidthD.getInt();
	if (renderHeightD.type() == DL::DT_Integer)
		rs.filmHeight = (uint32)renderHeightD.getInt();
	if (cropD.type() == DL::DT_Group) {
		const DL::DataGroup& crop = cropD.getGroup();
		if (crop.anonymousCount() == 4 && crop.isAllAnonymousNumber()) {
			rs.cropMinX = crop.at(0).getNumber();
			rs.cropMaxX = crop.at(1).getNumber();
			rs.cropMinY = crop.at(2).getNumber();
			rs.cropMaxY = crop.at(3).getNumber();
		}
	}
	if (spectralDomainD.isNumber()) {
		rs.spectralStart = spectralDomainD.getNumber();
		rs.spectralEnd	 = rs.spectralStart;
		rs.spectralMono	 = true;
	} else if (spectralDomainD.type() == DL::DT_Group) {
		const DL::DataGroup& sd = spectralDomainD.getGroup();
		if (sd.anonymousCount() == 2 && sd.isAllAnonymousNumber()) {
			rs.spectralStart = sd.at(0).getNumber();
			rs.spectralEnd	 = sd.at(1).getNumber();
			if (rs.spectralEnd < rs.spectralStart)
				std::swap(rs.spectralStart, rs.spectralEnd);
			rs.spectralMono = rs.spectralStart == rs.spectralEnd;
		}
	}
	if (spectralHeroD.type() == DL::DT_Bool)
		rs.spectralHero = spectralHeroD.getBool();
	std::vector<DL::DataGroup> inner;
	for (size_t i = 0; i < top.anonymousCount(); ++i)
		if (top.at(i).type() == DL::DT_Group)
			inner.push_back(top.at(i).getGroup());
	SceneLoadContext ctx(env.get(), path);
	setupEnvironment(inner, ctx);
	return env;
}

void SceneLoader::setupEnvironment(const std::vector<DL::DataGroup>& groups, SceneLoadContext& ctx)
{ // SceneLoader.cpp:154-190
	for (const DL::DataGroup& entry : groups) {
		const std::string& id = entry.id();
		if (id == "scene")
			PR_LOG(L_ERROR) << "[Loader] Invalid inner scene entry" << std::endl;
		else if (id == "include")
			addInclude(entry, ctx);
		else if (id == "sampler")
			addSampler(entry, ctx);
		else if (id == "filter")
			addFilter(entry, ctx);
		else if (id == "integrator")
			addIntegrator(entry, ctx);
		else if (id == "texture") // "just a sophisticated node", SceneLoader.cpp:167-168
			addTexture(entry, ctx);
		else if (id == "node")
			addNode(entry, ctx);
		else if (id == "mesh")
			addMesh(entry, ctx);
		else if (id == "graph" || id == "embed")
			addSubGraph(entry, ctx);
		else if (id == "material")
			addMaterial(entry, ctx);
		else if (id == "emission")
			addEmission(entry, ctx);
		else if (id == "entity")
			addEntity(entry, nullptr, ctx);
		else if (id == "light")
			addLight(entry, ctx);
		else if (id == "camera")
			addCamera(entry, ctx);
		else if (id == "spectral_mapper")
			addSpectralMapper(entry, ctx);
		else if (id == "output")
			ctx.environment()->outputSpecification().parse(entry); // SceneLoader.cpp: OutputSpecification::parse
	}
}

static bool typeOf(const DL::DataGroup& g, const char* what, std::string& type)
{
	const DL::Data typeD = g.getFromKey("type");
	if (typeD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "[Loader] " << what << " could not be load. No valid type given." << std::endl;
		return false;
	}
	type = lower(typeD.getString());
	return true;
}

void SceneLoader::addSampler(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:192-260
	std::string type;
	if (!typeOf(group, "Sampler", type))
		return;
	const DL::Data slotD = group.getFromKey("slot");
	std::string slot	 = slotD.type() == DL::DT_String ? lower(slotD.getString()) : "aa";
	auto fac			 = ctx.environment()->samplerManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown sampler type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto sampler	 = fac->create(type, ctx);
	if (!sampler) {
		PR_LOG(L_ERROR) << "[Loader] Could not create sampler of type " << type << std::endl;
		return;
	}
	RenderSettings& rs = ctx.environment()->renderSettings();
	if (slot == "aa" || slot == "pixel" || slot == "antialiasing")
		rs.aaSamplerFactory = sampler;
	else if (slot == "lens")
		rs.lensSamplerFactory = sampler;
	else if (slot == "time")
		rs.timeSamplerFactory = sampler;
	else if (slot == "spectral" || slot == "spectrum")
		rs.spectralSamplerFactory = sampler;
	else
		PR_LOG(L_ERROR) << "[Loader] Unknown sampler slot " << slot << std::endl;
}
void SceneLoader::addFilter(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	std::string type;
	if (!typeOf(group, "Filter", type))
		return;
	auto fac = ctx.environment()->filterManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown filter type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto filter		 = fac->create(type, ctx);
	if (filter)
		ctx.environment()->renderSettings().pixelFilterFactory = filter;
}
void SceneLoader::addIntegrator(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	std::string type;
	if (!typeOf(group, "Integrator", type))
		return;
	auto fac = ctx.environment()->integratorManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown integrator type " << type << " (the device path has the 'direct' path tracer, 'ao' and 'visualfeedback')" << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto intgr		 = fac->create(type, ctx);
	if (!intgr) {
		PR_LOG(L_ERROR) << "[Loader] Could not create integrator of type " << type << std::endl;
		return;
	}
	if (ctx.environment()->renderSettings().integratorFactory)
		PR_LOG(L_WARNING) << "[Loader] Integrator already selected. Replacing it " << std::endl;
	ctx.environment()->renderSettings().integratorFactory = intgr;
}
void SceneLoader::addSpectralMapper(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	std::string type;
	if (!typeOf(group, "Spectral mapper", type))
		return;
	const DL::Data purposeD = group.getFromKey("purpose");
	const std::string purpose = purposeD.type() == DL::DT_String ? lower(purposeD.getString()) : "pixel";
	auto fac				  = ctx.environment()->spectralMapperManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown spectral mapper type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto m			 = fac->create(type, ctx);
	if (m)
		ctx.environment()->renderSettings().spectralMapperFactories[purpose] = m;
}

Transformf SceneLoader::extractTransform(const DL::DataGroup& group)
{ // SceneLoader.cpp:386-444 + parser/MathParser.cpp
	const DL::Data transformD = group.getFromKey("transform");
	const DL::Data posD		  = group.getFromKey("position");
	const DL::Data rotD		  = group.getFromKey("rotation");
	const DL::Data scaleD	  = group.getFromKey("scale");
	auto getVector			  = [](const DL::DataGroup& arr, bool& ok) {
		   Vector3f res(0, 0, 0);
		   ok = false;
		   if ((arr.anonymousCount() == 2 || arr.anonymousCount() == 3) && arr.isAllAnonymousNumber()) {
			   res = Vector3f(arr.at(0).getNumber(), arr.at(1).getNumber(), arr.anonymousCount() == 3 ? arr.at(2).getNumber() : 0.0f);
			   ok  = true;
		   }
		   return res;
	};
	Transformf t;
	if (transformD.type() == DL::DT_Group) {
		const DL::DataGroup& g = transformD.getGroup();
		if (g.isAllAnonymousNumber() && g.anonymousCount() == 16) {
			for (int i = 0; i < 3; ++i) {
				for (int j = 0; j < 3; ++j)
					t.L(i, j) = g.at(i * 4 + j).getNumber();
				t.T[i] = g.at(i * 4 + 3).getNumber();
			}
		} else if (g.isAllAnonymousNumber() && g.anonymousCount() == 9) {
			for (int i = 0; i < 3; ++i)
				for (int j = 0; j < 3; ++j)
					t.L(i, j) = g.at(i * 3 + j).getNumber();
		} else {
			PR_LOG(L_WARNING) << "Couldn't set transform " << std::endl;
		}
		return t;
	}
	bool ok		 = true;
	Vector3f pos = Vector3f(0, 0, 0), sca = Vector3f(1, 1, 1);
	Matrix3f rot;
	if (posD.type() == DL::DT_Group) {
		pos = getVector(posD.getGroup(), ok);
		if (!ok)
			PR_LOG(L_WARNING) << "Couldn't set position " << std::endl;
	}
	if (ok && rotD.type() == DL::DT_Group) {
		const DL::DataGroup& g = rotD.getGroup();
		if (g.isArray() && g.anonymousCount() == 4 && g.isAllAnonymousNumber()) {
			rot = quaternionToMatrix(g.at(0).getNumber(), g.at(1).getNumber(), g.at(2).getNumber(), g.at(3).getNumber());
		} else if (g.id() == "euler" && g.anonymousCount() == 3 && g.isAllAnonymousNumber()) {
			const float x = g.at(0).getNumber() * PR_PI / 180, y = g.at(1).getNumber() * PR_PI / 180, z = g.at(2).getNumber() * PR_PI / 180;
			Matrix3f rx, ry, rz; // az * ay * ax
			rx(1, 1) = std::cos(x);
			rx(1, 2) = -std::sin(x);
			rx(2, 1) = std::sin(x);
			rx(2, 2) = std::cos(x);
			ry(0, 0) = std::cos(y);
			ry(0, 2) = std::sin(y);
			ry(2, 0) = -std::sin(y);
			ry(2, 2) = std::cos(y);
			rz(0, 0) = std::cos(z);
			rz(0, 1) = -std::sin(z);
			rz(1, 0) = std::sin(z);
			rz(1, 1) = std::cos(z);
			rot		 = rz * ry * rx;
		} else {
			ok = false;
			PR_LOG(L_WARNING) << "Couldn't set rotation " << std::endl;
		}
	}
	if (ok && scaleD.isNumber()) {
		const float s = scaleD.getNumber();
		sca			  = Vector3f(s, s, s);
	} else if (ok && scaleD.type() == DL::DT_Group) {
		sca = getVector(scaleD.getGroup(), ok);
		if (!ok)
			PR_LOG(L_WARNING) << "Couldn't set scale " << std::endl;
	}
	if (!ok)
		return Transformf::Identity();
	for (int i = 0; i < 3; ++i)
		for (int j = 0; j < 3; ++j)
			t.L(i, j) = rot(i, j) * sca[j]; // fromPositionOrientationScale: R * diag(s)
	t.T = pos;
	return t;
}

void SceneLoader::addEntity(const DL::DataGroup& group, const ITransformable* parent, SceneLoadContext& ctx)
{ // SceneLoader.cpp:446-510
	const DL::Data nameD	 = group.getFromKey("name");
	const std::string name	 = nameD.type() == DL::DT_String ? nameD.getString() : "UNKNOWN";
	std::string type;
	if (!typeOf(group, "Entity", type))
		return;
	auto fac = ctx.environment()->entityManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown entity type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	ctx.transform()	 = parent ? parent->transform() * extractTransform(group) : extractTransform(group);
	auto entity		 = fac->create(type, ctx);
	if (!entity) {
		PR_LOG(L_ERROR) << "[Loader] Could not create entity of type " << type << std::endl;
		return;
	}
	auto vis = [&](const char* k, uint32 bit) {
		const DL::Data d = group.getFromKey(k);
		return (d.type() != DL::DT_Bool || d.getBool()) ? bit : 0u;
	};
	entity->setVisibilityFlags(vis("camera_visible", PRB_RAY_CAMERA) | vis("light_visible", PRB_RAY_LIGHT) | vis("bounce_visible", PRB_RAY_BOUNCE)
							   | vis("shadow_visible", PRB_RAY_SHADOW));
	ctx.environment()->sceneDatabase()->Entities.add(name, entity);
	for (size_t i = 0; i < group.anonymousCount(); ++i)
		if (group.at(i).type() == DL::DT_Group && group.at(i).getGroup().id() == "entity")
			addEntity(group.at(i).getGroup(), entity.get(), ctx);
}
void SceneLoader::addCamera(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:512-556
	const DL::Data typeD = group.getFromKey("type");
	std::string type	 = "standard";
	if (typeD.type() == DL::DT_String)
		type = lower(typeD.getString());
	else if (typeD.isValid()) {
		PR_LOG(L_ERROR) << "[Loader] No valid camera type set" << std::endl;
		return;
	}
	auto fac = ctx.environment()->cameraManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown camera type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	ctx.transform()	 = extractTransform(group);
	auto camera		 = fac->create(type, ctx);
	if (!camera) {
		PR_LOG(L_ERROR) << "[Loader] Could not create camera of type " << type << std::endl;
		return;
	}
	if (ctx.environment()->activeCamera)
		PR_LOG(L_WARNING) << "[Loader] Active camera already exists. Replacing it " << type << std::endl;
	ctx.environment()->activeCamera = camera;
}
void SceneLoader::addLight(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	std::string type;
	if (!typeOf(group, "Light", type))
		return;
	auto fac = ctx.environment()->infiniteLightManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown infinite light type " << type << " ('sky'/'sun' are SURVEY 8(f)-1 'next' rows)" << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	ctx.transform()	 = extractTransform(group);
	auto light		 = fac->create(type, ctx);
	if (!light) {
		PR_LOG(L_ERROR) << "[Loader] Could not create light of type " << type << std::endl;
		return;
	}
	ctx.environment()->sceneDatabase()->InfiniteLights.add(light);
}
void SceneLoader::addEmission(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	const DL::Data nameD   = group.getFromKey("name");
	const std::string name = nameD.type() == DL::DT_String ? nameD.getString() : "UNKNOWN";
	std::string type	   = "standard";
	const DL::Data typeD   = group.getFromKey("type");
	if (typeD.type() == DL::DT_String)
		type = lower(typeD.getString());
	if (ctx.environment()->sceneDatabase()->Emissions.has(name)) {
		PR_LOG(L_ERROR) << "[Loader] Emission name already exists." << std::endl;
		return;
	}
	auto fac = ctx.environment()->emissionManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown emission type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto ems		 = fac->create(type, ctx);
	if (!ems) {
		PR_LOG(L_ERROR) << "[Loader] Could not create emission of type " << type << std::endl;
		return;
	}
	ctx.environment()->sceneDatabase()->Emissions.add(name, ems);
}
void SceneLoader::addMaterial(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	const DL::Data nameD   = group.getFromKey("name");
	const std::string name = nameD.type() == DL::DT_String ? nameD.getString() : "UNKNOWN";
	std::string type;
	if (!typeOf(group, "Material", type))
		return;
	if (ctx.environment()->sceneDatabase()->Materials.has(name)) {
		PR_LOG(L_ERROR) << "[Loader] Material name already exists." << std::endl;
		return;
	}
	auto fac = ctx.environment()->materialManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown material type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto mat		 = fac->create(type, ctx);
	if (!mat) {
		PR_LOG(L_ERROR) << "[Loader] Could not create material of type " << type << std::endl;
		return;
	}
	mat->setID((uint32)ctx.environment()->sceneDatabase()->Materials.size());
	ctx.environment()->sceneDatabase()->Materials.add(name, mat);
}
void SceneLoader::addNode(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // named node: (node :name 'x' :type 'refl' ...)
	const DL::Data nameD = group.getFromKey("name");
	if (nameD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "[Loader] Node has no name" << std::endl;
		return;
	}
	std::string type;
	if (!typeOf(group, "Node", type))
		return;
	auto fac = ctx.environment()->nodeManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown node type " << type << std::endl;
		return;
	}
	ctx.parameters() = populateObjectParameters(group, ctx);
	auto node		 = fac->create(type, ctx);
	if (node)
		ctx.environment()->namedNodes[nameD.getString()] = node;
}
void SceneLoader::addTexture(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:656-670 + parser/TextureParser.cpp:64-211
	const DL::Data nameD = group.getFromKey("name");
	if (nameD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "[Loader] No texture name set" << std::endl;
		return;
	}
	const std::string name = nameD.getString();
	DL::Data fileD		   = group.getFromKey("file");
	if (!fileD.isValid())
		fileD = group.getFromKey("filename");
	if (fileD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "No valid filename given for texture " << name << std::endl;
		return;
	}
	auto parseWrap = [](std::string w) { // TextureParser.cpp:20-32; WrapDefault of a file without a wrap attribute is black
		w = lower(w);
		return w == "clamp" ? PRB_WRAP_CLAMP : w == "periodic" ? PRB_WRAP_PERIODIC : w == "mirror" ? PRB_WRAP_MIRROR : PRB_WRAP_BLACK;
	};
	int wrapS = PRB_WRAP_BLACK, wrapT = PRB_WRAP_BLACK;
	const DL::Data wrapD = group.getFromKey("wrap");
	if (wrapD.type() == DL::DT_String) {
		wrapS = wrapT = parseWrap(wrapD.getString());
	} else if (wrapD.type() == DL::DT_Group) {
		const DL::DataGroup arr = wrapD.getGroup();
		if (arr.anonymousCount() > 0 && arr.at(0).type() == DL::DT_String)
			wrapS = parseWrap(arr.at(0).getString());
		if (arr.anonymousCount() > 1 && arr.at(1).type() == DL::DT_String)
			wrapT = parseWrap(arr.at(1).getString());
	}
	int interp			   = PRB_TEX_BICUBIC; // InterpSmartBicubic without derivatives magnifies: bicubic (TextureParser.cpp:50-60)
	const DL::Data interpD = group.getFromKey("interpolation");
	if (interpD.type() == DL::DT_String) {
		const std::string i = lower(interpD.getString());
		interp				= i == "closest" ? PRB_TEX_CLOSEST : (i == "bi" || i == "bilinear") ? PRB_TEX_BILINEAR : PRB_TEX_BICUBIC;
	}
	const DL::Data mipD = group.getFromKey("mip");
	if (mipD.type() == DL::DT_String && lower(mipD.getString()) != "none")
		PR_LOG(L_WARNING) << "Texture " << name << ": MIP levels are not used on this path (lookups carry no derivatives, ImageNode.cpp:143-145)" << std::endl;
	std::string type	 = "color";
	const DL::Data typeD = group.getFromKey("type");
	if (typeD.type() == DL::DT_String)
		type = lower(typeD.getString());
	else
		PR_LOG(L_WARNING) << "No valid type given for texture " << name << ": Assuming color" << std::endl;
	if (ctx.environment()->namedNodes.count(name)) {
		PR_LOG(L_ERROR) << "Texture " << name << " already exists" << std::endl;
		return;
	}
	if (type != "grayscale" && type != "color" && type != "spectral") {
		PR_LOG(L_ERROR) << (type == "scalar" ? "Scalar textures are not supported on this path: texture " : "No known type given for texture ") << name << std::endl;
		return;
	}
	const std::string file = ctx.setupParametricPath(fileD.getString());
	auto node			   = makeImageNode(file, interp, wrapS, wrapT, ctx.environment()->defaultSpectralUpsampler());
	if (node)
		ctx.environment()->namedNodes[name] = node;
}
uint32 SceneLoader::addNodeInline(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp: inline shading network, node type == group id
	const std::string type = lower(group.id());
	auto fac			   = ctx.environment()->nodeManager.getFactory(type);
	if (!fac) {
		PR_LOG(L_ERROR) << "[Loader] Unknown node type " << type << std::endl;
		return P_INVALID_REFERENCE;
	}
	SceneLoadContext sub = ctx;
	sub.parameters()	 = populateObjectParameters(group, ctx);
	auto node			 = fac->create(type, sub);
	if (!node) {
		PR_LOG(L_ERROR) << "[Loader] Could not create node of type " << type << std::endl;
		return P_INVALID_REFERENCE;
	}
	return ctx.environment()->sceneDatabase()->Nodes.add(node);
}

void SceneLoader::addMesh(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp addMesh + parser/MeshParser.cpp:135-247
	const DL::Data nameD = group.getFromKey("name");
	if (nameD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "[Loader] Mesh has no name" << std::endl;
		return;
	}
	auto me	 = std::make_shared<MeshBase>();
	me->name = nameD.getString();
	auto loadAttribute = [](const DL::DataGroup& grp, int D, std::vector<float>& arr) {
		arr.reserve(grp.anonymousCount() * D);
		for (size_t j = 0; j < grp.anonymousCount(); ++j) {
			const DL::Data& d = grp.at(j);
			if (d.type() != DL::DT_Group || (int)d.getGroup().anonymousCount() != D || !d.getGroup().isAllAnonymousNumber())
				return false;
			for (int k = 0; k < D; ++k)
				arr.push_back(d.getGroup().at(k).getNumber());
		}
		return true;
	};
	for (size_t i = 0; i < group.anonymousCount(); ++i) {
		if (group.at(i).type() != DL::DT_Group) {
			PR_LOG(L_ERROR) << "Invalid entry in mesh description." << std::endl;
			return;
		}
		const DL::DataGroup& grp = group.at(i).getGroup();
		if (grp.id() == "attribute") {
			const DL::Data t = grp.getFromKey("type");
			if (t.type() != DL::DT_String) {
				PR_LOG(L_ERROR) << "Mesh attribute has no valid type." << std::endl;
				return;
			}
			bool ok = true;
			if (t.getString() == "p")
				ok = loadAttribute(grp, 3, me->vertices);
			else if (t.getString() == "n")
				ok = loadAttribute(grp, 3, me->normals);
			else if (t.getString() == "t" || t.getString() == "uv")
				ok = loadAttribute(grp, 2, me->uvs);
			else if (t.getString() == "w" || t.getString() == "dp" || t.getString() == "u")
				PR_LOG(L_WARNING) << "Mesh attribute '" << t.getString() << "' is not used by the device path." << std::endl;
			else {
				PR_LOG(L_ERROR) << "Unknown mesh attribute '" << t.getString() << "'." << std::endl;
				return;
			}
			if (!ok) {
				PR_LOG(L_ERROR) << "Mesh attribute '" << t.getString() << "' is invalid." << std::endl;
				return;
			}
		}
	}
	for (size_t i = 0; i < group.anonymousCount(); ++i) {
		const DL::DataGroup& grp = group.at(i).getGroup();
		if (grp.id() == "faces") {
			me->indices.reserve(grp.anonymousCount() * 4);
			for (size_t j = 0; j < grp.anonymousCount(); ++j) {
				const DL::Data& d = grp.at(j);
				if (d.type() != DL::DT_Group || !d.getGroup().isAllAnonymousOfType(DL::DT_Integer)
					|| (d.getGroup().anonymousCount() != 3 && d.getGroup().anonymousCount() != 4)) {
					PR_LOG(L_ERROR) << "Only triangle or quads allowed in mesh faces." << std::endl;
					return;
				}
				const DL::DataGroup& f = d.getGroup();
				for (size_t k = 0; k < 4; ++k)
					me->indices.push_back(k < f.anonymousCount() ? (uint32)f.at(k).getInt() : PR_INVALID_ID);
			}
		} else if (grp.id() == "normal_faces" || grp.id() == "texture_faces") {
			PR_LOG(L_ERROR) << "Separate '" << grp.id() << "' index sets are not supported on the device path." << std::endl;
			return;
		} else if (grp.id() == "materials") {
			for (size_t j = 0; j < grp.anonymousCount(); ++j) {
				if (grp.at(j).type() != DL::DT_Integer || grp.at(j).getInt() < 0) {
					PR_LOG(L_ERROR) << "Given index is invalid." << std::endl;
					return;
				}
				me->materialSlots.push_back((uint32)grp.at(j).getInt());
			}
		}
	}
	std::string err;
	if (!me->isValid(&err)) {
		PR_LOG(L_ERROR) << "Loaded mesh is invalid: " << err << std::endl;
		return;
	}
	ctx.environment()->meshes[me->name] = me;
}

// Wavefront OBJ -> MeshBase.  The reference goes through tinyobjloader with triangulate = true
// (src/loader/archives/WavefrontLoader.cpp:24-200): all shapes of the file are merged into one mesh, polygons become
// triangles (tinyobj clips ears starting at the first corner, which for the convex polygons of the example data is the
// fan (0,k,k+1)), materials are ignored.  tinyobj keeps one index list per attribute; the device mesh layout has one shared
// index list, so corners are merged by their (v, vn, vt) triple -- same positions, normals and uvs at every face corner,
// same face order and therefore the same primitive ids.
static bool loadWavefront(const std::string& file, bool flipNormal, MeshBase& mesh)
{
	std::ifstream in(file);
	if (!in) {
		PR_LOG(L_ERROR) << "Wavefront file: Could not open file " << file << std::endl;
		return false;
	}
	std::vector<float> P, N, T;
	struct Corner {
		int v, n, t;
		bool operator<(const Corner& o) const { return std::tie(v, n, t) < std::tie(o.v, o.n, o.t); }
	};
	std::vector<std::vector<Corner>> polygons;
	std::string line;
	while (std::getline(in, line)) {
		std::istringstream ls(line);
		std::string tag;
		if (!(ls >> tag) || tag[0] == '#')
			continue;
		if (tag == "v" || tag == "vn") {
			float x = 0, y = 0, z = 0;
			ls >> x >> y >> z;
			std::vector<float>& dst = tag == "v" ? P : N;
			dst.insert(dst.end(), { x, y, z });
		} else if (tag == "vt") {
			float u = 0, v = 0;
			ls >> u >> v;
			T.insert(T.end(), { u, v });
		} else if (tag == "f") {
			std::vector<Corner> poly;
			std::string tok;
			while (ls >> tok) {
				// v | v/vt | v//vn | v/vt/vn ; 1-based, negative = relative to the elements read so far
				int idx[3]	  = { 0, 0, 0 };
				int field	  = 0;
				size_t start  = 0;
				for (size_t i = 0; i <= tok.size() && field < 3; ++i)
					if (i == tok.size() || tok[i] == '/') {
						if (i > start)
							idx[field] = std::atoi(tok.substr(start, i - start).c_str());
						++field;
						start = i + 1;
					}
				auto fix = [](int i, size_t count) { return i > 0 ? i - 1 : (i < 0 ? (int)count + i : -1); };
				poly.push_back(Corner{ fix(idx[0], P.size() / 3), fix(idx[2], N.size() / 3), fix(idx[1], T.size() / 2) });
			}
			if (poly.size() >= 3)
				polygons.push_back(std::move(poly));
		}
	}
	if (P.empty() || polygons.empty()) {
		PR_LOG(L_ERROR) << "Wavefront file: No vertices or faces given in " << file << std::endl;
		return false;
	}
	const bool hasN = !N.empty(), hasT = !T.empty();
	std::map<Corner, uint32> merged;
	auto cornerIndex = [&](Corner c) {
		c.v = std::max(0, c.v);
		c.n = hasN ? std::max(0, c.n) : -1;
		c.t = hasT ? std::max(0, c.t) : -1;
		auto it = merged.find(c);
		if (it != merged.end())
			return it->second;
		const uint32 id = (uint32)mesh.vertexCount();
		if ((size_t)c.v * 3 + 2 >= P.size() || (hasN && (size_t)c.n * 3 + 2 >= N.size()) || (hasT && (size_t)c.t * 2 + 1 >= T.size()))
			return PR_INVALID_ID;
		mesh.vertices.insert(mesh.vertices.end(), P.begin() + 3 * c.v, P.begin() + 3 * c.v + 3);
		if (hasN)
			for (int k = 0; k < 3; ++k)
				mesh.normals.push_back(flipNormal ? -N[3 * c.n + k] : N[3 * c.n + k]);
		if (hasT)
			mesh.uvs.insert(mesh.uvs.end(), T.begin() + 2 * c.t, T.begin() + 2 * c.t + 2);
		merged.emplace(c, id);
		return id;
	};
	for (const auto& poly : polygons)
		for (size_t k = 1; k + 1 < poly.size(); ++k) {
			const uint32 tri[3] = { cornerIndex(poly[0]), cornerIndex(poly[k]), cornerIndex(poly[k + 1]) };
			if (tri[0] == PR_INVALID_ID || tri[1] == PR_INVALID_ID || tri[2] == PR_INVALID_ID) {
				PR_LOG(L_ERROR) << "Wavefront file: face index out of range in " << file << std::endl;
				return false;
			}
			mesh.indices.insert(mesh.indices.end(), { tri[0], tri[1], tri[2], PR_INVALID_ID });
		}
	return true;
}

void SceneLoader::addSubGraph(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:773-846
	const DL::Data loaderD = group.getFromKey("loader");
	const DL::Data fileD   = group.getFromKey("file");
	if (fileD.type() != DL::DT_String) {
		PR_LOG(L_ERROR) << "[Loader] Could not get file for subgraph entry." << std::endl;
		return;
	}
	std::string loader;
	if (loaderD.type() == DL::DT_String) {
		loader = loaderD.getString();
	} else {
		PR_LOG(L_WARNING) << "[Loader] No valid loader set. Assuming 'obj'." << std::endl;
		loader = "obj";
	}
	if (loader != "obj") { // 'ply' and 'mts' archives: not needed by the path's configurations
		PR_LOG(L_ERROR) << "[Loader] Unknown " << loader << " loader." << std::endl;
		return;
	}
	const std::string file	 = ctx.setupParametricPath(fileD.getString());
	const DL::Data nameD	 = group.getFromKey("name");
	const DL::Data flipD	 = group.getFromKey("flipNormal");
	auto me					 = std::make_shared<MeshBase>();
	if (!loadWavefront(file, flipD.type() == DL::DT_Bool && flipD.getBool(), *me))
		return;
	me->name = nameD.type() == DL::DT_String ? nameD.getString() : file;
	if (ctx.environment()->meshes.count(me->name))
		PR_LOG(L_ERROR) << "Mesh " << me->name << " already in use." << std::endl;
	std::string err;
	if (!me->isValid(&err)) {
		PR_LOG(L_WARNING) << "Obj file could not construct a valid mesh data: " << err << std::endl;
		return;
	}
	ctx.environment()->meshes[me->name] = me;
}

void SceneLoader::addInclude(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:848-886
	if (group.anonymousCount() == 1 && group.at(0).type() == DL::DT_String) {
		const std::string real = ctx.setupParametricPath(group.at(0).getString());
		std::vector<DL::DataGroup> groups;
		try {
			groups = DL::parseFile(real);
		} catch (const std::exception& e) {
			PR_LOG(L_ERROR) << "[Loader] Could not include " << real << ": " << e.what() << std::endl;
			return;
		}
		ctx.pushFile(real);
		setupEnvironment(groups, ctx);
		ctx.popFile();
	} else {
		PR_LOG(L_ERROR) << "[Loader] Invalid include" << std::endl;
	}
}

static bool valueToParameter(const DL::Data& entry, SceneLoadContext& ctx, Parameter& out,
							 const std::function<Parameter(const DL::DataGroup&, SceneLoadContext&)>& unpack)
{ // one arm of populateObjectParameters, SceneLoader.cpp:888-997
	switch (entry.type()) {
	case DL::DT_Integer: out = Parameter::fromInt(entry.getInt()); return true;
	case DL::DT_Float: out = Parameter::fromNumber(entry.getNumber()); return true;
	case DL::DT_Bool: out = Parameter::fromBool(entry.getBool()); return true;
	case DL::DT_String: out = Parameter::fromString(entry.getString()); return true;
	case DL::DT_Group: {
		const DL::DataGroup& grp = entry.getGroup();
		if (grp.isArray()) {
			const size_t n = grp.anonymousCount();
			if (grp.isAllAnonymousOfType(DL::DT_Bool)) {
				std::vector<bool> arr(n);
				for (size_t i = 0; i < n; ++i)
					arr[i] = grp.at(i).getBool();
				out = Parameter::fromBoolArray(arr);
			} else if (grp.isAllAnonymousOfType(DL::DT_Integer)) {
				std::vector<int64> arr(n);
				for (size_t i = 0; i < n; ++i)
					arr[i] = grp.at(i).getInt();
				out = Parameter::fromIntArray(arr);
			} else if (grp.isAllAnonymousNumber()) {
				std::vector<float> arr(n);
				for (size_t i = 0; i < n; ++i)
					arr[i] = grp.at(i).getNumber();
				out = Parameter::fromNumberArray(arr);
			} else if (grp.isAllAnonymousOfType(DL::DT_String)) {
				std::vector<std::string> arr(n);
				for (size_t i = 0; i < n; ++i)
					arr[i] = grp.at(i).getString();
				out = Parameter::fromStringArray(arr);
			} else {
				PR_LOG(L_ERROR) << "[Loader] Array inner type mismatch" << std::endl;
				return false;
			}
			return true;
		}
		out = unpack(grp, ctx);
		return out.isValid();
	}
	default: PR_LOG(L_ERROR) << "[Loader] Invalid parameter entry value." << std::endl; return false;
	}
}
ParameterGroup SceneLoader::populateObjectParameters(const DL::DataGroup& group, SceneLoadContext& ctx)
{
	ParameterGroup params;
	Parameter p;
	for (const auto& entry : group.getNamedEntries())
		if (valueToParameter(entry, ctx, p, &SceneLoader::unpackShadingNetwork))
			params.addParameter(entry.key(), p);
	for (const auto& entry : group.getAnonymousEntries()) {
		// child objects (entity children, mesh attribute blocks ...) are not parameters of their parent
		if (entry.type() == DL::DT_Group && !entry.getGroup().isArray()) {
			const std::string& id = entry.getGroup().id();
			if (id == "entity" || id == "attribute" || id == "faces" || id == "materials" || id == "channel")
				continue;
		}
		if (valueToParameter(entry, ctx, p, &SceneLoader::unpackShadingNetwork))
			params.addParameter(p);
	}
	return params;
}
Parameter SceneLoader::unpackShadingNetwork(const DL::DataGroup& group, SceneLoadContext& ctx)
{ // SceneLoader.cpp:999-1041
	if (group.id() == "texture" || group.id() == "node") {
		if (group.anonymousCount() == 1 && group.at(0).type() == DL::DT_String) {
			const auto node = ctx.getRawNode(group.at(0).getString());
			if (node)
				return Parameter::fromReference(ctx.environment()->sceneDatabase()->Nodes.add(node));
			PR_LOG(L_ERROR) << "[Loader] Unknown " << group.id() << " " << group.at(0).getString() << std::endl;
		} else {
			PR_LOG(L_ERROR) << "[Loader] Invalid " << group.id() << " parameter" << std::endl;
		}
	} else if (group.id() == "deg2rad") {
		if (group.anonymousCount() == 1 && group.at(0).isNumber())
			return Parameter::fromNumber(group.at(0).getNumber() * PR_DEG2RAD);
		PR_LOG(L_ERROR) << "[Loader] Invalid node parameter" << std::endl;
	} else if (group.id() == "rad2deg") {
		if (group.anonymousCount() == 1 && group.at(0).isNumber())
			return Parameter::fromNumber(group.at(0).getNumber() * PR_RAD2DEG);
		PR_LOG(L_ERROR) << "[Loader] Invalid node parameter" << std::endl;
	} else {
		const uint32 id = addNodeInline(group, ctx);
		if (id != P_INVALID_REFERENCE)
			return Parameter::fromReference(id);
	}
	return Parameter();
}

// ------------------------------------------------------------------ LightSampler
LightSampler::LightSampler(const SceneDatabase& db, float sceneRadius, const SpectralRange& cameraRange)
	: mLightSpectralRange(cameraRange)
{ // LightSampler.cpp:11-132
	const float scene_area = 2 * PR_PI * sceneRadius;
	const auto& entities   = db.Entities.getAll();
	const auto& emissions  = db.Emissions.getAll();
	const auto& inflights  = db.InfiniteLights.getAll();
	size_t light_count	   = inflights.size();
	for (const auto& e : entities)
		if (e->hasEmission())
			++light_count;
	if (light_count == 0)
		return;
	const SpectralBlob test_wvl_distr(0.05f, 0.05f + 0.3f, 0.05f + 0.6f, 0.95f); // SpectralBlob::LinSpaced(0.05, 0.95)
	std::vector<float> intensities;
	for (const auto& e : entities) {
		if (!e->hasEmission() || e->emissionID() >= emissions.size())
			continue;
		const IEmission* emission	= emissions[e->emissionID()].get();
		const SpectralRange range	= emission->spectralRange().bounded(cameraRange);
		SpectralBlob test_wvl;
		for (int i = 0; i < 4; ++i)
			test_wvl[i] = range.Start + range.span() * test_wvl_distr[i];
		const float area	  = e->worldSurfaceArea();
		const float intensity = area * emission->power(test_wvl).mean();
		mEmissiveSurfaceArea += area;
		mEmissiveSurfacePower += intensity;
		PR_LOG(L_INFO) << "(Area) Light '" << e->name() << "' Area " << area << "m2 Intensity " << intensity << "W [" << range.Start << ", " << range.End << "]" << std::endl;
		intensities.push_back(intensity);
		mLightSpectralRange += range;
	}
	mEmissivePower = mEmissiveSurfacePower;
	for (const auto& infL : inflights) {
		const SpectralRange range = infL->spectralRange().bounded(cameraRange);
		SpectralBlob test_wvl;
		for (int i = 0; i < 4; ++i)
			test_wvl[i] = range.Start + range.span() * test_wvl_distr[i];
		const float intensity = scene_area * infL->power(test_wvl).mean();
		mEmissivePower += intensity;
		PR_LOG(L_INFO) << "(Inf) Light '" << infL->name() << "' Area " << scene_area << "m2 Intensity " << intensity << "W" << std::endl;
		intensities.push_back(intensity);
		mLightSpectralRange += range;
	}
	float full = 0;
	mSelector  = Distribution1D(intensities.size());
	mSelector.generate([&](size_t i) { return intensities[i]; }, &full);
	if (full <= PR_EPSILON) {
		PR_LOG(L_WARNING) << "Lights are available but seems like they have no power" << std::endl;
	} else {
		const float invI = 1 / full;
		for (float& f : intensities)
			f *= invI;
	}
	size_t k = 0;
	for (const auto& e : entities) {
		if (!e->hasEmission() || e->emissionID() >= emissions.size())
			continue;
		Light l;
		l.id			  = (uint32)mLights.size();
		l.entity		  = e.get();
		l.emission		  = emissions[e->emissionID()].get();
		l.relContribution = intensities[k++];
		mLights.push_back(l);
	}
	for (const auto& infL : inflights) {
		Light l;
		l.id			  = (uint32)mLights.size();
		l.infLight		  = infL.get();
		l.relContribution = intensities[k++];
		mLights.push_back(l);
	}
	if (mEmissivePower <= PR_EPSILON)
		mInfLightSelectionProbability = inflights.empty() ? 0.0f : 0.5f;
	else
		mInfLightSelectionProbability = (mEmissivePower - mEmissiveSurfacePower) / mEmissivePower;
}
} // namespace PR
