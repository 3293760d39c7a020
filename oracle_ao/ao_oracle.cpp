// ORACLE of the 'ao' integrator -- test infrastructure only (the checker, never the product).  A scalar CPU restatement of the
// semantics documented at prb_set_integrator (include/prb200_abi.h), built from the oracle's existing pieces: constructCameraRay,
// traceScene (closest and any hit), Integrator::makeIP / nextRay / pushSpectralFragment, cos_hemi and the film fold of
// orc_render_lpe.  One pcg32_fast stream per pixel, drawn in sample order: camera, then u2, u1 per occlusion ray.
#include "../oracle/oracle.cpp"

namespace {
void renderAOSample(Integrator& I, uint32_t px, uint32_t py, uint32_t iteration, Rng& rnd, uint32_t sampleCount)
{
	Film& film = I.film;
	Stats& stats = I.stats;
	stats.c[S_PIXEL_SAMPLE]++;
	CameraSampleOut cs;
	constructCameraRay(I.sc, px, py, iteration, rnd, cs);
	I.grp.importance  = cs.importance;
	I.grp.wvl		  = cs.wvl;
	I.grp.wvlPDF	  = cs.wvlPDF;
	I.grp.blendWeight = cs.blendWeight;
	RayS ray;
	ray.O	  = cs.origin;
	ray.D	  = cs.dir;
	ray.tmin  = cs.tmin;
	ray.tmax  = cs.tmax;
	ray.wvl	  = cs.wvl;
	ray.depth = 0;
	ray.flags = (cs.mono ? PRB_RAY_MONOCHROME : 0) | PRB_RAY_CAMERA;
	stats.c[S_CAMERA_RAY]++;
	stats.c[S_PRIMARY]++;
	Hit h;
	const bool hit = traceScene(I.sc, I.A, ray.O, ray.D, ray.tmin, ray.tmax, false, h);
	ray.D		   = normalized(ray.D); // RayStream::getRay re-normalises on read, RayStream.cpp:167
	// the MIS weight of handleZero (direct.cpp:415-464 with Throughput 1): also the weight of the occlusion fragment
	const Blob heroFactor = (ray.flags & PRB_RAY_MONOCHROME) ? heroOnly() : blob(1);
	const Blob mis		  = heroFactor / (cs.wvlPDF * bsum(heroFactor));
	if (!hit) {
		stats.c[S_BG_HIT]++;
		I.pushSpectralFragment(mis, blob(1), blob(0), ray.flags);
		return;
	}
	IP ip;
	I.makeIP(ray, h, ip); // N is not flipped toward the viewer
	stats.c[S_ENTITY_HIT]++;
	stats.c[S_CAMERA_DEPTH]++;
	const uint32_t p = I.pixelIndex;
	film.sampleCount[p] += 1; // the first-hit part of handleCameraVertex (pushSPFragment -> commitShadingPoints)
	if (film.aov) {
		float* a = film.aov + 10 * (size_t)p;
		a[0] += ip.N.x;
		a[1] += ip.N.y;
		a[2] += ip.N.z;
		a[3] += ip.P.x;
		a[4] += ip.P.y;
		a[5] += ip.P.z;
		a[6] += ip.g.u;
		a[7] += ip.g.v;
		a[8] += std::sqrt(ip.depth2);
		a[9] += (float)ip.g.entity;
	}
	if (film.aovExt) {
		float* b = film.aovExt + PRB_AOV_EXT * (size_t)p;
		b[0] += ip.Nx.x;
		b[1] += ip.Nx.y;
		b[2] += ip.Nx.z;
		b[3] += ip.Ny.x;
		b[4] += ip.Ny.y;
		b[5] += ip.Ny.z;
		b[6] += ip.ray.D.x;
		b[7] += ip.ray.D.y;
		b[8] += ip.ray.D.z;
		b[9] += (float)ip.g.material;
		b[10] += (float)ip.g.emission;
	}
	uint32_t occluded = 0;
	for (uint32_t j = 0; j < sampleCount; ++j) {
		const float u2	   = rnd.getFloat(); // cos_hemi(rnd.getFloat(), rnd.getFloat()) evaluated right to left
		const float u1	   = rnd.getFloat();
		const V3 dir	   = fromTangentSpace(ip.N, ip.Nx, ip.Ny, cos_hemi(u1, u2));
		const RayS occRay = I.nextRay(ip, dir, PRB_RAY_BOUNCE, 0.0001f, PR_INF);
		stats.c[S_SHADOW]++;
		Hit oh;
		if (traceScene(I.sc, I.A, occRay.O, occRay.D, occRay.tmin, occRay.tmax, true, oh))
			++occluded;
	}
	const float d = 1.0f - (float)occluded / (float)sampleCount;
	I.pushSpectralFragment(mis, blob(1), blob(d), ray.flags);
}
} // namespace

extern "C" {
// orc_render_lpe (without expression channels, lpe_mean must be NULL) for the 'ao' integrator with sample_count occlusion rays
void orc_render_ao(orc_scene* s, uint64_t* rng, const prb_tile* tiles, size_t n_tiles, uint32_t first_iteration, uint32_t iteration_count,
				   float* film_mean, uint32_t* sample_count, float* aov, uint64_t* stats11, int threads, uint32_t* feedback, float* online_mean,
				   float* online_variance, float* lpe_mean, float* aov_ext, uint32_t ao_sample_count)
{
	(void)lpe_mean;
	const prb_settings& st = s->sc.d->settings;
	const uint32_t W	   = st.film_width;
	Film film;
	film.iterXYZ.assign((size_t)W * st.film_height * 3, 0.0f);
	film.mean		 = film_mean;
	film.sampleCount = sample_count;
	film.aov		 = aov;
	film.aovExt		 = aov_ext;
	film.feedback	 = feedback;
	film.varMean	 = online_mean;
	film.varVar		 = online_variance;
	std::vector<uint32_t> pixels;
	for (size_t t = 0; t < n_tiles; ++t)
		for (uint32_t y = tiles[t].sy; y < tiles[t].ey; ++y)
			for (uint32_t x = tiles[t].sx; x < tiles[t].ex; ++x)
				pixels.push_back(y * W + x);
	threads = std::max(1, threads);
	std::vector<Stats> tstats(threads);
	std::atomic<size_t> cursor{ 0 };
	auto worker = [&](int tid) {
		setFTZ();
		Integrator I{ s->sc, s->accel, film, tstats[tid], 0, Group{} };
		for (;;) {
			const size_t begin = cursor.fetch_add(256);
			if (begin >= pixels.size())
				break;
			const size_t end = std::min(pixels.size(), begin + 256);
			for (size_t i = begin; i < end; ++i) {
				const uint32_t p = pixels[i];
				Rng rnd{ rng[p] };
				for (uint32_t it = first_iteration; it < first_iteration + iteration_count; ++it) {
					I.pixelIndex = p;
					for (int c = 0; c < 3; ++c)
						film.iterXYZ[3 * (size_t)p + c] = 0.0f;
					renderAOSample(I, p % W, p / W, it, rnd, ao_sample_count);
					const float iter = (float)(it + 1); // FrameOutputDevice::onEndOfIteration, as orc_render_lpe
					for (int c = 0; c < 3; ++c) {
						float& a = film.mean[3 * (size_t)p + c];
						a		 = (a * (float)it + film.iterXYZ[3 * (size_t)p + c]) / iter;
					}
					if (film.varMean && film.varVar)
						for (int c = 0; c < 3; ++c) {
							const float value = film.iterXYZ[3 * (size_t)p + c];
							float& mean		  = film.varMean[3 * (size_t)p + c];
							float& var		  = film.varVar[3 * (size_t)p + c];
							const float delta = value - mean;
							mean += delta / iter;
							const float delta2 = value - mean;
							var				   = (var * (float)it + delta * delta2) / iter;
						}
				}
				rng[p] = rnd.s;
			}
		}
	};
	std::vector<std::thread> pool;
	for (int t = 1; t < threads; ++t)
		pool.emplace_back(worker, t);
	worker(0);
	for (auto& th : pool)
		th.join();
	if (stats11)
		for (int t = 0; t < threads; ++t)
			for (int i = 0; i < 11; ++i)
				stats11[i] += tstats[t].c[i];
}
}
