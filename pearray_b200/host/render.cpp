// Render driver: the host half of reference RenderContext::start / RenderThread::main
// (src/core/renderer/RenderContext.cpp:65-139, RenderThread.cpp:36-70).  One RenderContext drives one GPU
// through the C ABI; ranks of a multi-GPU job own interleaved tiles (tile_id % worldSize == rank).
#include "prh.h"

namespace PR {
RenderContext::RenderContext(const std::shared_ptr<Environment>& env, int device, uint32 rank, uint32 worldSize)
	: mEnv(env)
	, mRank(rank)
	, mWorldSize(std::max(1u, worldSize))
{
	SceneCompiler compiler(env.get());
	mScene = compiler.compile();
	if (!mScene)
		return;
	mIntegrator = env->renderSettings().integratorFactory->createInstance();
	if (prb_create(device, &mCtx) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_create failed: " << prb_last_error() << std::endl;
		mCtx = nullptr;
		return;
	}
	if (prb_upload_scene(mCtx, &mScene->desc) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_upload_scene failed: " << prb_last_error() << std::endl;
		prb_destroy(mCtx);
		mCtx = nullptr;
		return;
	}
	if (prb_set_integrator(mCtx, &mScene->integrator) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_set_integrator failed: " << prb_last_error() << std::endl;
		prb_destroy(mCtx);
		mCtx = nullptr;
	}
}
RenderContext::~RenderContext()
{
	if (mCtx)
		prb_destroy(mCtx);
}

bool RenderContext::start(uint32 rtx, uint32 rty, uint32 iterations)
{
	if (!mCtx)
		return false;
	const prb_settings& st = mScene->desc.settings;
	if (iterations == 0)
		iterations = st.max_sample_count;
	// RenderRandomMap (RenderContext.cpp:84)
	const std::vector<uint64> rng = buildRenderRandomMap(st.seed, st.film_width, st.film_height, settings().progressive ? 128 : st.max_sample_count);
	if (prb_upload_rng(mCtx, rng.data(), rng.size()) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_upload_rng failed: " << prb_last_error() << std::endl;
		return false;
	}
	prb_film_clear(mCtx);
	// RenderTileMap::init (RenderContext.cpp:91); interleaved ownership across ranks (SURVEY 8(e))
	const std::vector<RenderTile> tiles = buildTileMap(st.view_x, st.view_y, st.view_w, st.view_h, rtx, rty);
	mOwnedTiles.clear();
	for (size_t i = 0; i < tiles.size(); ++i)
		if (i % mWorldSize == mRank)
			mOwnedTiles.push_back(tiles[i]);
	mIntegrator->onInit(this);
	mIntegrator->onStart();
	auto instance = mIntegrator->createThreadInstance(this, 0);
	instance->onStart();
	// The reference walks iteration by iteration, tile by tile (RenderThread.cpp:44-66 calling onTile).  All
	// tiles of this rank and all iterations go to the device as ONE batch: a pixel's samples only depend on the
	// pixel's own RNG stream, so the order across pixels is free (bit-identical results).
	std::vector<prb_tile> pt;
	for (const RenderTile& t : mOwnedTiles)
		pt.push_back(prb_tile{ t.sx, t.sy, t.ex, t.ey });
	bool ok = true;
	if (!pt.empty() && prb_render_tiles(mCtx, pt.data(), pt.size(), 0, iterations) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_render_tiles failed: " << prb_last_error() << std::endl;
		ok = false;
	}
	instance->onEnd();
	mIntegrator->onEnd();
	// interleaved tiles: every pixel was rendered by exactly one rank, the reduced film on rank 0 is bit-identical to a
	// single-GPU render (collective: every rank of the communicator gets here, also one that owns no tile)
	if (ok && mHasCommunicator && prb_film_reduce_comm(mCtx, PRB_PARTITION_TILES, iterations, 0) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_film_reduce_comm failed: " << prb_last_error() << std::endl;
		ok = false;
	}
	return ok;
}
bool RenderContext::joinCommunicator(const uint8_t id[PRB_COMM_UNIQUE_ID_BYTES])
{
	if (!mCtx)
		return false;
	if (prb_comm_init(mCtx, id, (int)mRank, (int)mWorldSize) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_comm_init failed: " << prb_last_error() << std::endl;
		return false;
	}
	mHasCommunicator = true;
	return true;
}
bool RenderContext::combineFilms(const std::vector<RenderContext*>& contexts)
{
	std::vector<prb_ctx*> ctxs;
	for (RenderContext* rc : contexts) {
		if (!rc || !rc->mCtx)
			return false;
		ctxs.push_back(rc->mCtx);
	}
	if (prb_film_reduce(ctxs.data(), (int)ctxs.size(), PRB_PARTITION_TILES) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_film_reduce failed: " << prb_last_error() << std::endl;
		return false;
	}
	return true;
}
void RenderContext::waitForFinish()
{
	if (mCtx)
		prb_sync(mCtx);
}
std::vector<float> RenderContext::filmXYZ()
{
	const prb_settings& st = mScene->desc.settings;
	std::vector<float> xyz((size_t)st.film_width * st.film_height * 3);
	if (mCtx && prb_film_download(mCtx, xyz.data(), nullptr) != PRB_OK)
		PR_LOG(L_ERROR) << "prb_film_download failed: " << prb_last_error() << std::endl;
	return xyz;
}
int RenderContext::saveOutputs(const std::string& workingDir)
{ // Environment::save -> OutputSpecification::save (reference src/loader/Environment.cpp, OutputSpecification.cpp:439-464)
	const prb_settings& st = mScene->desc.settings;
	const size_t n		   = (size_t)st.film_width * st.film_height;
	std::vector<float> xyz(n * 3), aov;
	std::vector<uint32> count(n), feedback(n);
	if (!mCtx || prb_film_download(mCtx, xyz.data(), count.data()) != PRB_OK) {
		PR_LOG(L_ERROR) << "prb_film_download failed: " << prb_last_error() << std::endl;
		return -1;
	}
	FilmView film;
	film.width = film.fullWidth = st.film_width;
	film.height = film.fullHeight = st.film_height;
	film.xyz					  = xyz.data();
	film.sampleCount			  = count.data();
	aov.resize(n * 10);
	if (prb_film_download_aov(mCtx, aov.data()) == PRB_OK) // AOVs are optional (prb_settings.enable_aov)
		film.aov = aov.data();
	std::vector<float> aovExt;
	if (st.want_aov_ext) {
		aovExt.resize(n * PRB_AOV_EXT);
		if (prb_film_download_aov_ext(mCtx, aovExt.data()) == PRB_OK)
			film.aovExt = aovExt.data();
	}
	if (prb_film_download_feedback(mCtx, feedback.data()) == PRB_OK)
		film.feedback = feedback.data();
	std::vector<float> onlineMean, onlineVariance;
	if (st.want_variance) {
		onlineMean.resize(n * 3);
		onlineVariance.resize(n * 3);
		if (prb_film_download_variance(mCtx, onlineMean.data(), onlineVariance.data()) == PRB_OK) {
			film.onlineMean		= onlineMean.data();
			film.onlineVariance = onlineVariance.data();
		}
	}
	std::vector<std::vector<float>> lpe(mScene->desc.n_lpe, std::vector<float>(n * 3));
	for (uint32 k = 0; k < mScene->desc.n_lpe; ++k)
		film.lpe.push_back(prb_film_download_lpe(mCtx, k, lpe[k].data()) == PRB_OK ? lpe[k].data() : nullptr);
	return mEnv->outputSpecification().save(workingDir, film, mRank);
}
prb_stats RenderContext::statistics() const
{
	prb_stats s{};
	if (mCtx)
		prb_get_stats(mCtx, &s);
	return s;
}

// IMaterial::eval / ::sample through the device (unit-level entry points of the C ABI)
void IMaterial::eval(const MaterialEvalInput& in, MaterialEvalOutput& out, const RenderTileSession& session) const
{
	prb_material_query q{};
	for (int i = 0; i < 3; ++i) {
		q.V[i] = in.V[i];
		q.L[i] = in.L[i];
	}
	for (int i = 0; i < 4; ++i)
		q.wavelength_nm[i] = in.WavelengthNM[i];
	q.uv[0]		  = in.UV.x;
	q.uv[1]		  = in.UV.y;
	q.ray_flags	  = in.RayFlags;
	q.material_id = mID;
	prb_material_result r{};
	if (prb_material_eval(session.context()->deviceContext(), &q, 1, &r) != PRB_OK)
		PR_LOG(L_ERROR) << "prb_material_eval failed: " << prb_last_error() << std::endl;
	for (int i = 0; i < 4; ++i) {
		out.Weight[i] = r.weight[i];
		out.PDF_S[i]  = r.pdf_s[i];
	}
	out.Flags = r.flags;
	out.Type  = (MaterialScatteringType)r.type;
}
void IMaterial::sample(const MaterialSampleInput& in, MaterialSampleOutput& out, const RenderTileSession& session) const
{
	prb_material_query q{};
	for (int i = 0; i < 3; ++i)
		q.V[i] = in.V[i];
	for (int i = 0; i < 4; ++i)
		q.wavelength_nm[i] = in.WavelengthNM[i];
	q.uv[0]		  = in.UV.x;
	q.uv[1]		  = in.UV.y;
	q.ray_flags	  = in.RayFlags;
	q.material_id = mID;
	q.rng_state	  = in.RND ? in.RND->state() : 3;
	prb_material_result r{};
	if (prb_material_sample(session.context()->deviceContext(), &q, 1, &r) != PRB_OK)
		PR_LOG(L_ERROR) << "prb_material_sample failed: " << prb_last_error() << std::endl;
	for (int i = 0; i < 4; ++i) {
		out.IntegralWeight[i] = r.weight[i];
		out.PDF_S[i]		  = r.pdf_s[i];
	}
	out.L	  = Vector3f(r.L[0], r.L[1], r.L[2]);
	out.Flags = r.flags;
	out.Type  = (MaterialScatteringType)r.type;
	if (in.RND)
		in.RND->setState(r.rng_state);
}
} // namespace PR
