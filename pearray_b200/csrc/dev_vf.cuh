// Kernel of the visual-feedback integrator ('vf', prb_set_integrator with PRB_INTEGRATOR_VF): the debug view of scene set-up.
// Per pixel sample: the camera ray of 'direct' (same draws), its closest hit and, on a hit, one linear-sRGB colour chosen by the
// mode (entity, material, emission or primitive id through a palette; uv; front/back face; |N.D|).  The colour goes into the film
// as XYZ = M c (M: sRGB D65 RGB -> XYZ), past the spectral fragment path: the image has no spectral noise and the sRGB tone mode
// of the film gives c back.  A miss folds a zero sample, as under 'ao'.
//
//   one VF iteration = one sample for every owned pixel = 1 kernel (k_vf, slot = thread), so every iteration is a full wave.
//   k_vf exists for the small-scene path (flat scene in shared memory, traverseSmall) and for the BVH (traverseScene).  The mode
//   is a kernel argument: the switch is warp-uniform and the build keeps two instantiations.
#pragma once
#include "dev_ao.cuh"

namespace prb {
// palette(id): a golden-ratio hue sequence (consecutive ids get distant hues, no table wraps) at S = 0.7, V = 0.9 through the
// textbook HSV -> RGB.  Plain fp32 operations, each rounded (the build has -fmad=false): the oracle and the tests restate it
// bit for bit.
PRB_DEV V3 vfPalette(uint32_t id)
{
	const float x  = (float)id * 0.618034f;
	const float h6 = 6.0f * (x - floorf(x));
	const float i  = floorf(h6);
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
PRB_DEV V3 vfPaletteOrBlack(uint32_t id) { return id == PRB_INVALID_ID ? mk(0, 0, 0) : vfPalette(id); }

// the colour of a hit (D: the normalised camera direction)
PRB_DEV V3 vfColour(uint32_t mode, const GeomPoint& g, const V3& D)
{
	switch (mode) {
	case PRB_VF_MATERIAL_ID: return vfPaletteOrBlack(g.material);
	case PRB_VF_EMISSION_ID: return vfPaletteOrBlack(g.emission);
	case PRB_VF_PRIMITIVE_ID: return vfPalette(g.prim);
	case PRB_VF_PARAMETER: return mk(g.u, g.v, 0);
	case PRB_VF_INSIDE: return dot(D, g.N) > 0 ? mk(1, 0, 0) : mk(0, 1, 0);
	case PRB_VF_NDOTV: {
		const float a = fabsf(dot(g.N, D));
		return mk(a, a, a);
	}
	default: return vfPalette(g.entity);
	}
}

template <bool SMALL>
__global__ void __launch_bounds__(128) k_vf(const __grid_constant__ DScene S, WFState W, uint32_t mode)
{
	__shared__ uint4 smallScene[SMALL ? SMALL_SCENE_U4 : 1];
	const uint32_t slot	   = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t endIter = W.counters[CNT_END_ITER];
	uint32_t pix = 0, it = endIter;
	if (slot < W.nSlots) {
		pix = W.pixel[slot];
		it	= W.iter[slot];
	}
	if (SMALL) {
		for (uint32_t i = threadIdx.x; i < S.nSmallU4; i += blockDim.x)
			smallScene[i] = __ldg(S.small + i);
		__syncthreads();
	}
	const bool live = it < endIter;
	if (!__any_sync(0xFFFFFFFFu, live)) // (warp-uniform; no barrier follows) the pixels of the warp have all their samples
		return;
	Rng rnd{ 0 };
	CameraSampleOut cs;
	cs.origin = mk(0, 0, 0);
	cs.dir	  = mk(0, 0, 1);
	cs.tmin = cs.tmax = 0;
	cs.mono			  = false;
	if (live) {
		rnd = Rng{ W.rng[pix] };
		constructCameraRay(S, pix % S.settings.film_width, pix / S.settings.film_width, it, rnd, cs);
	}
	HitRec h;
	bool found;
	if (SMALL)
		found = traverseSmall(smallScene, S.nSmallEnts, S.nSmallFaces, live, false, cs.origin, cs.dir, cs.tmin, cs.tmax, h);
	else
		found = traverseScene(S, live, false, cs.origin, cs.dir, cs.tmin, cs.tmax, h);
	bool hit	 = false;
	uint32_t sBg = 0;
	if (live) {
		W.iter[slot] = it + 1;
		V3 c		 = mk(0, 0, 0);
		if (!found) { // a zero fragment, which can only leave feedback bits (as k_ao_primary)
			++sBg;
			const bool groupMono  = S.settings.spectral_mono || !S.settings.spectral_hero;
			const uint32_t flags  = PRB_RAY_CAMERA | (cs.mono ? PRB_RAY_MONOCHROME : 0u);
			const Blob heroFactor = cs.mono ? heroOnly() : blob(1);
			const uint32_t fb	  = fragmentBitsZeroRadiance(S, heroFactor / (cs.wvlPDF * bsum(heroFactor)), blob(1), flags, groupMono);
			if (fb)
				W.feedback[pix] |= fb;
		} else { // makeIP: RayStream::getRay re-normalises the camera ray on read, RayStream.cpp:167
			const V3 D = normalized(cs.dir);
			const V3 P = cs.origin + h.t * D;
			GeomPoint g;
			provideGeometryPointBody(S, h.entity, h.prim, h.u, h.v, P, g);
			addCameraVertex(W, pix, g, P, D, norm2(cs.origin - P)); // as 'direct' at path length 1
			c	= vfColour(mode, g, D);
			hit = true;
		}
		// XYZ = M c, M the inverse of the film's sRGB tone matrix (ToneMapper / RGBConverter::fromXYZ), rounded to fp32
		foldSampleIntoFilm(W, pix, (4.123907387e-01f * c.x + 3.575841486e-01f * c.y) + 1.804806888e-01f * c.z,
						   (2.126389146e-01f * c.x + 7.151684165e-01f * c.y) + 7.219225168e-02f * c.z,
						   (1.933080330e-02f * c.x + 1.191947088e-01f * c.y) + 9.505316615e-01f * c.z, it + 1);
		W.rng[pix] = rnd.s;
	}
	{
		const uint32_t s = live ? 1u : 0u, e = hit ? 1u : 0u;
		const int which[6]	   = { ST_PIXEL_SAMPLE, ST_CAMERA_RAY, ST_PRIMARY, ST_ENTITY_HIT, ST_CAMERA_DEPTH, ST_BG_HIT };
		const uint32_t vals[6] = { s, s, s, e, e, sBg };
		statAddMany(W.stats, which, vals);
	}
}

__global__ void __launch_bounds__(128) k_vf_begin(WFState W) { beginFirstHitRender(W, blockIdx.x * blockDim.x + threadIdx.x); }
} // namespace prb
