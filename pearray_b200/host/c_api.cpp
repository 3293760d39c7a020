// Flat C entry points over the C++ host layer, for ctypes (tests, bench.py) and other FFI users.
// They expose the loader, the compiled POD scene and the render driver; nothing here computes samples.
#include "prh.h"

using namespace PR;

namespace {
struct SceneHandle {
	std::shared_ptr<Environment> env;
	std::shared_ptr<CompiledScene> scene;
};
thread_local std::string g_err;
} // namespace

namespace PR {
double hosekSkyRadiance(double solarElevation, double turbidity, double albedo, double theta, double gamma, double wavelength);
void sunElevationAzimuth(int year, int month, int day, int hour, int minute, float seconds, float latitude, float longitude, float timezone, float* elevation,
						 float* azimuth);
float sunRadiance(float wavelength, float theta, float turbidity);
}

extern "C" {
// sky / sun host models (skysun.cpp), exposed for the known-answer tests
double prh_hosek_sky_radiance(double solar_elevation, double turbidity, double albedo, double theta, double gamma, double wavelength)
{
	try {
		return hosekSkyRadiance(solar_elevation, turbidity, albedo, theta, gamma, wavelength);
	} catch (const std::exception& e) {
		g_err = e.what();
		return -1.0;
	}
}
void prh_sun_position(int year, int month, int day, int hour, int minute, float seconds, float latitude, float longitude, float timezone, float* elevation,
					  float* azimuth)
{
	sunElevationAzimuth(year, month, day, hour, minute, seconds, latitude, longitude, timezone, elevation, azimuth);
}
float prh_sun_radiance(float wavelength, float theta, float turbidity) { return sunRadiance(wavelength, theta, turbidity); }

const char* prh_last_error() { return g_err.c_str(); }
void prh_set_verbosity(int level) { logVerbosity() = level; }
// LightPathExpression(expr).isValid() / .match(path): tokens = n (type, event) pairs; returns -1 invalid, 0 no match, 1 match
int prh_lpe_match(const char* expr, const int32_t* tokens, uint32_t n)
{
	const LPEAutomaton a = compileLPE(expr ? expr : "");
	if (!a.valid)
		return -1;
	std::vector<std::pair<int, int>> t;
	for (uint32_t i = 0; i < n; ++i)
		t.emplace_back(tokens[2 * i], tokens[2 * i + 1]);
	return a.match(t) ? 1 : 0;
}
// sizeof() of the POD structs of include/prb200_abi.h as this library was compiled, for checking FFI mirrors (ctypes, cgo ...)
uint32_t prh_abi_sizeof(const char* name)
{
	const std::string n = name ? name : "";
#define PRH_SIZE_OF(T) \
	if (n == #T)       \
		return (uint32_t)sizeof(T);
	PRH_SIZE_OF(prb_ray_soa)
	PRH_SIZE_OF(prb_hit_soa)
	PRH_SIZE_OF(prb_node)
	PRH_SIZE_OF(prb_material)
	PRH_SIZE_OF(prb_emission)
	PRH_SIZE_OF(prb_mesh)
	PRH_SIZE_OF(prb_entity)
	PRH_SIZE_OF(prb_bvh8_node)
	PRH_SIZE_OF(prb_bvh_tri)
	PRH_SIZE_OF(prb_light)
	PRH_SIZE_OF(prb_sampler)
	PRH_SIZE_OF(prb_spectral_mapper)
	PRH_SIZE_OF(prb_camera)
	PRH_SIZE_OF(prb_settings)
	PRH_SIZE_OF(prb_scene_desc)
	PRH_SIZE_OF(prb_lpe)
	PRH_SIZE_OF(prb_tile)
	PRH_SIZE_OF(prb_stats)
	PRH_SIZE_OF(prb_material_query)
	PRH_SIZE_OF(prb_material_result)
	PRH_SIZE_OF(prb_integrator)
#undef PRH_SIZE_OF
	return 0;
}

// Load a .prc file (or source string) and compile it; returns NULL on error.
void* prh_load_scene_file(const char* path)
{
	auto env = SceneLoader::loadFromFile(path);
	if (!env) {
		g_err = std::string("could not load scene ") + path;
		return nullptr;
	}
	SceneCompiler c(env.get());
	auto scene = c.compile();
	if (!scene) {
		g_err = "could not compile scene";
		return nullptr;
	}
	return new SceneHandle{ env, scene };
}
void* prh_load_scene_string(const char* source, const char* virtual_path)
{
	auto env = SceneLoader::loadFromString(source, virtual_path ? virtual_path : "");
	if (!env) {
		g_err = "could not load scene from string";
		return nullptr;
	}
	SceneCompiler c(env.get());
	auto scene = c.compile();
	if (!scene) {
		g_err = "could not compile scene";
		return nullptr;
	}
	return new SceneHandle{ env, scene };
}
void* prh_make_soup(uint32_t triangles, uint64_t seed, uint32_t film_w, uint32_t film_h)
{
	return new SceneHandle{ nullptr, makeSoupScene(triangles, seed, film_w, film_h) };
}
// (output ...) blocks of the scene: number of files, and <dir>/results[_index]/<name>.exr written from host film buffers
// (xyz: 3 floats / pixel, count: 1 u32 / pixel, aov: 10 floats / pixel or NULL), as prb_film_download / prb_film_aov return them
uint32_t prh_output_file_count(void* h)
{
	auto* s = static_cast<SceneHandle*>(h);
	return s->env ? (uint32_t)s->env->outputSpecification().files().size() : 0u;
}
int prh_save_outputs(void* h, const char* dir, const float* xyz, const uint32_t* count, const float* aov, uint32_t context_index)
{
	auto* s = static_cast<SceneHandle*>(h);
	if (!s->env) {
		g_err = "scene has no loader environment (synthetic scene)";
		return -1;
	}
	const prb_settings& st = s->scene->desc.settings;
	FilmView film;
	film.width		 = st.film_width;
	film.height		 = st.film_height;
	film.fullWidth	 = st.film_width;
	film.fullHeight	 = st.film_height;
	film.xyz		 = xyz;
	film.sampleCount = count;
	film.aov		 = aov;
	return s->env->outputSpecification().save(dir ? dir : "", film, context_index);
}
void prh_free_scene(void* h) { delete static_cast<SceneHandle*>(h); }
const prb_scene_desc* prh_scene_desc(void* h) { return &static_cast<SceneHandle*>(h)->scene->desc; }
// the prb_integrator record of the scene's (integrator ...) block; PRB_ERR_INVALID_ARG for a null argument
int prh_scene_integrator(void* h, prb_integrator* out)
{
	if (!h || !out) {
		g_err = "null argument";
		return PRB_ERR_INVALID_ARG;
	}
	*out = static_cast<SceneHandle*>(h)->scene->integrator;
	return PRB_OK;
}
prb_scene_desc* prh_scene_desc_mutable(void* h) { return &static_cast<SceneHandle*>(h)->scene->desc; }
double prh_scene_bvh_seconds(void* h) { return static_cast<SceneHandle*>(h)->scene->bvhBuildSeconds; }
float prh_scene_radius(void* h) { return static_cast<SceneHandle*>(h)->scene->sceneRadius; }
// override the iteration budget (reference sampleCountOverride); re-describes nothing, only the setting
void prh_scene_set_spp(void* h, uint32_t spp) { static_cast<SceneHandle*>(h)->scene->desc.settings.max_sample_count = spp; }

// RenderRandomMap states (film_w * film_h uint64)
void prh_build_rng_map(uint64_t seed, uint32_t w, uint32_t h, uint32_t rng_delta, uint64_t* out)
{
	const auto v = buildRenderRandomMap(seed, w, h, rng_delta);
	std::memcpy(out, v.data(), v.size() * sizeof(uint64_t));
}
// tile map; returns the tile count (writes at most capacity tiles)
uint32_t prh_build_tile_map(uint32_t vx, uint32_t vy, uint32_t vw, uint32_t vh, uint32_t rtx, uint32_t rty, prb_tile* out, uint32_t capacity)
{
	const auto t = buildTileMap(vx, vy, vw, vh, rtx, rty);
	for (uint32_t i = 0; i < t.size() && i < capacity; ++i)
		out[i] = prb_tile{ t[i].sx, t[i].sy, t[i].ex, t[i].ey };
	return (uint32_t)t.size();
}

// --- small host-logic probes used by the CPU test-suite
int prh_upsample_rgb(const float* rgb, float* coeffs)
{
	try {
		Environment env;
		env.defaultSpectralUpsampler()->prepare(&rgb[0], &rgb[1], &rgb[2], &coeffs[0], &coeffs[1], &coeffs[2], 1);
		return 0;
	} catch (const std::exception& e) {
		g_err = e.what();
		return -1;
	}
}
void prh_upsample_eval(const float* coeffs, const float* wavelengths, float* out, uint32_t n)
{
	SpectralUpsampler::computeSingle(coeffs[0], coeffs[1], coeffs[2], wavelengths, out, n);
}
float prh_cie_eval(int channel, float wavelength)
{
	return channel == 0 ? CIE::eval_x(wavelength) : (channel == 1 ? CIE::eval_y(wavelength) : CIE::eval_z(wavelength));
}
void prh_random_stream(uint64_t seed, uint32_t n, uint32_t* out32, float* outf)
{
	Random r(seed);
	for (uint32_t i = 0; i < n; ++i) {
		Random c		 = r;
		const uint32_t v = r.get32();
		if (out32)
			out32[i] = v;
		if (outf)
			outf[i] = c.getFloat();
	}
}
uint64_t prh_random_advance(uint64_t state, uint64_t delta)
{
	Random r(0);
	r.setState(state);
	r.advance(delta);
	return r.state();
}
// sampler probe: generate2D / generate1D of the scene's AA sampler from a fresh Random(seed)
void prh_list_plugins(void* h, char* buf, uint32_t cap)
{
	std::string s;
	Environment* env = static_cast<SceneHandle*>(h)->env.get();
	if (env) {
		auto add = [&](const char* kind, const std::vector<std::string>& names) {
			s += kind;
			s += ":";
			for (const auto& n : names)
				s += " " + n;
			s += "\n";
		};
		add("integrator", env->integratorManager.names());
		add("material", env->materialManager.names());
		add("emission", env->emissionManager.names());
		add("entity", env->entityManager.names());
		add("camera", env->cameraManager.names());
		add("infinitelight", env->infiniteLightManager.names());
		add("sampler", env->samplerManager.names());
		add("filter", env->filterManager.names());
		add("spectralmapper", env->spectralMapperManager.names());
		add("node", env->nodeManager.names());
	}
	std::snprintf(buf, cap, "%s", s.c_str());
}

// --- render driver (RenderContext) for FFI users
void* prh_render_context_create(void* scene, int device, uint32_t rank, uint32_t world)
{
	SceneHandle* h = static_cast<SceneHandle*>(scene);
	if (!h->env) {
		g_err = "render context needs a loaded scene";
		return nullptr;
	}
	auto* rc = new RenderContext(h->env, device, rank, world);
	if (!rc->valid()) {
		g_err = std::string("render context creation failed: ") + prb_last_error();
		delete rc;
		return nullptr;
	}
	return rc;
}
int prh_render_context_start(void* rc, uint32_t rtx, uint32_t rty, uint32_t iterations)
{
	return static_cast<RenderContext*>(rc)->start(rtx, rty, iterations) ? 0 : -1;
}
int prh_render_context_save_outputs(void* rc, const char* dir) { return static_cast<RenderContext*>(rc)->saveOutputs(dir ? dir : ""); }
void prh_render_context_wait(void* rc) { static_cast<RenderContext*>(rc)->waitForFinish(); }
prb_ctx* prh_render_context_device(void* rc) { return static_cast<RenderContext*>(rc)->deviceContext(); }
void prh_render_context_destroy(void* rc) { delete static_cast<RenderContext*>(rc); }
int prh_render_context_join_communicator(void* rc, const uint8_t* id128) { return static_cast<RenderContext*>(rc)->joinCommunicator(id128) ? 0 : -1; }
int prh_render_contexts_combine(void** rcs, int n)
{
	std::vector<RenderContext*> v;
	for (int i = 0; i < n; ++i)
		v.push_back(static_cast<RenderContext*>(rcs[i]));
	return RenderContext::combineFilms(v) ? 0 : -1;
}
}
