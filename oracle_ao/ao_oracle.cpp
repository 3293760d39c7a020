// ORACLE of the integrators whose samples end at the first hit, 'ao' and 'visualfeedback' -- test infrastructure only (the
// checker, never the product).  Scalar CPU restatements of the semantics documented at prb_set_integrator
// (include/prb200_abi.h), built from the oracle's existing pieces: constructCameraRay, traceScene (closest and any hit),
// Integrator::makeIP / nextRay / pushSpectralFragment, cos_hemi and the film fold of orc_render_lpe.  One pcg32_fast stream per
// pixel, drawn in sample order: camera, then ('ao') u2, u1 per occlusion ray.
#include "../oracle/oracle.cpp"

namespace {
// the camera ray of 'direct' and its closest hit.  A miss pushes the zero fragment (MIS weight of handleZero, direct.cpp:415-464
// with Throughput 1) and returns false; a hit fills ip, counts it and adds the first-hit AOVs and the sample count (the first-hit
// part of handleCameraVertex: pushSPFragment -> commitShadingPoints).  mis: the weight of the miss fragment.
bool firstHit(Integrator& I, uint32_t px, uint32_t py, uint32_t iteration, Rng& rnd, IP& ip, Blob& mis)
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
	const Blob heroFactor = (ray.flags & PRB_RAY_MONOCHROME) ? heroOnly() : blob(1);
	mis					  = heroFactor / (cs.wvlPDF * bsum(heroFactor));
	if (!hit) {
		stats.c[S_BG_HIT]++;
		I.pushSpectralFragment(mis, blob(1), blob(0), ray.flags);
		return false;
	}
	I.makeIP(ray, h, ip); // N is not flipped toward the viewer
	stats.c[S_ENTITY_HIT]++;
	stats.c[S_CAMERA_DEPTH]++;
	const uint32_t p = I.pixelIndex;
	film.sampleCount[p] += 1;
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
	return true;
}

void renderAOSample(Integrator& I, uint32_t px, uint32_t py, uint32_t iteration, Rng& rnd, uint32_t sampleCount)
{
	IP ip;
	Blob mis; // also the weight of the occlusion fragment
	if (!firstHit(I, px, py, iteration, rnd, ip, mis))
		return;
	uint32_t occluded = 0;
	for (uint32_t j = 0; j < sampleCount; ++j) {
		const float u2	   = rnd.getFloat(); // cos_hemi(rnd.getFloat(), rnd.getFloat()) evaluated right to left
		const float u1	   = rnd.getFloat();
		const V3 dir	   = fromTangentSpace(ip.N, ip.Nx, ip.Ny, cos_hemi(u1, u2));
		const RayS occRay = I.nextRay(ip, dir, PRB_RAY_BOUNCE, 0.0001f, PR_INF);
		I.stats.c[S_SHADOW]++;
		Hit oh;
		if (traceScene(I.sc, I.A, occRay.O, occRay.D, occRay.tmin, occRay.tmax, true, oh))
			++occluded;
	}
	const float d = 1.0f - (float)occluded / (float)sampleCount;
	I.pushSpectralFragment(mis, blob(1), blob(d), ip.ray.flags);
}

// 'visualfeedback': palette(id) in plain fp32 (this build has -ffp-contract=off), h = frac(id * 0.618034), S = 0.7, V = 0.9,
// textbook HSV -> RGB
V3 vfPalette(uint32_t id)
{
	const float x  = (float)id * 0.618034f;
	const float h6 = 6.0f * (x - std::floor(x));
	const float i  = std::floor(h6);
	const float f  = h6 - i;
	const float S = 0.7f, V = 0.9f;
	const float p = V * (1.0f - S), q = V * (1.0f - S * f), t = V * (1.0f - S * (1.0f - f));
	switch ((int)i % 6) {
	case 0: return mk(V, t, p);
	case 1: return mk(q, V, p);
	case 2: return mk(p, V, t);
	case 3: return mk(p, q, V);
	case 4: return mk(t, p, V);
	default: return mk(V, p, q);
	}
}

void renderVFSample(Integrator& I, uint32_t px, uint32_t py, uint32_t iteration, Rng& rnd, uint32_t mode)
{
	IP ip;
	Blob mis;
	if (!firstHit(I, px, py, iteration, rnd, ip, mis))
		return;
	const GeomPoint& g = ip.g;
	const V3 D		   = ip.ray.D;
	V3 c;
	switch (mode) {
	case PRB_VF_MATERIAL_ID: c = g.material == PRB_INVALID_ID ? mk(0, 0, 0) : vfPalette(g.material); break;
	case PRB_VF_EMISSION_ID: c = g.emission == PRB_INVALID_ID ? mk(0, 0, 0) : vfPalette(g.emission); break;
	case PRB_VF_PRIMITIVE_ID: c = vfPalette(g.prim); break;
	case PRB_VF_PARAMETER: c = mk(g.u, g.v, 0); break;
	case PRB_VF_INSIDE: c = dot(D, g.N) > 0 ? mk(1, 0, 0) : mk(0, 1, 0); break;
	case PRB_VF_NDOTV: {
		const float a = std::fabs(dot(g.N, D));
		c			  = mk(a, a, a);
		break;
	}
	default: c = vfPalette(g.entity); break;
	}
	// XYZ = M c (sRGB D65 RGB -> XYZ in fp32), written to the film as it is: no spectral fragment, also on a monotonic film
	float* xyz = &I.film.iterXYZ[3 * (size_t)I.pixelIndex];
	xyz[0] += (4.123907387e-01f * c.x + 3.575841486e-01f * c.y) + 1.804806888e-01f * c.z;
	xyz[1] += (2.126389146e-01f * c.x + 7.151684165e-01f * c.y) + 7.219225168e-02f * c.z;
	xyz[2] += (1.933080330e-02f * c.x + 1.191947088e-01f * c.y) + 9.505316615e-01f * c.z;
}

// orc_render_lpe (without expression channels) for an integrator whose sample is sample(I, px, py, iteration, rnd)
template <class Sample>
void renderFirstHit(orc_scene* s, uint64_t* rng, const prb_tile* tiles, size_t n_tiles, uint32_t first_iteration, uint32_t iteration_count,
					float* film_mean, uint32_t* sample_count, float* aov, uint64_t* stats11, int threads, uint32_t* feedback, float* online_mean,
					float* online_variance, float* aov_ext, const Sample& sample)
{
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
					sample(I, p % W, p / W, it, rnd);
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
} // namespace

extern "C" {
// orc_render_lpe (without expression channels, lpe_mean must be NULL) for the 'ao' integrator with sample_count occlusion rays
void orc_render_ao(orc_scene* s, uint64_t* rng, const prb_tile* tiles, size_t n_tiles, uint32_t first_iteration, uint32_t iteration_count,
				   float* film_mean, uint32_t* sample_count, float* aov, uint64_t* stats11, int threads, uint32_t* feedback, float* online_mean,
				   float* online_variance, float* lpe_mean, float* aov_ext, uint32_t ao_sample_count)
{
	(void)lpe_mean;
	renderFirstHit(s, rng, tiles, n_tiles, first_iteration, iteration_count, film_mean, sample_count, aov, stats11, threads, feedback, online_mean,
				   online_variance, aov_ext, [&](Integrator& I, uint32_t px, uint32_t py, uint32_t it, Rng& rnd) { renderAOSample(I, px, py, it, rnd, ao_sample_count); });
}
// the same for the 'visualfeedback' integrator in mode vf_mode (PRB_VF_*)
void orc_render_vf(orc_scene* s, uint64_t* rng, const prb_tile* tiles, size_t n_tiles, uint32_t first_iteration, uint32_t iteration_count,
				   float* film_mean, uint32_t* sample_count, float* aov, uint64_t* stats11, int threads, uint32_t* feedback, float* online_mean,
				   float* online_variance, float* lpe_mean, float* aov_ext, uint32_t vf_mode)
{
	(void)lpe_mean;
	renderFirstHit(s, rng, tiles, n_tiles, first_iteration, iteration_count, film_mean, sample_count, aov, stats11, threads, feedback, online_mean,
				   online_variance, aov_ext, [&](Integrator& I, uint32_t px, uint32_t py, uint32_t it, Rng& rnd) { renderVFSample(I, px, py, it, rnd, vf_mode); });
}
}
