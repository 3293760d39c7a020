// Kernels of the ambient-occlusion integrator ('ao', prb_set_integrator with PRB_INTEGRATOR_AO).  Per pixel sample: the camera
// ray of 'direct' (same draws), its closest hit, then N cosine-weighted occlusion rays about the unflipped shading normal, each
// traced any-hit; the sample's value is 1 - occluded / N.  A miss folds a zero sample and counts no sample.
//
//   one AO iteration = one sample for every owned pixel = 3 kernels
//     k_ao_primary    per slot: camera ray, closest hit; on a hit the geometry point, the first-hit AOVs and the record the
//                     occlusion rays start from (P, N, Nx, Ny in vxP..vxNy, the RNG state after the camera draws); hit slots are
//                     appended to a list (warp-aggregated atomic).  Misses are folded into the film here.
//     k_ao_occlusion  persistent over the hits x N work items (count read from device memory).  Item (slot, j) finds its RNG
//                     state by jump-ahead: pcg32_fast is a pure MCG, so the state after the 2j draws of rays 0..j-1 is
//                     s * M^(2j) mod 2^64 (AOState::jump, computed by the host).  No direction buffer, and an occluded item adds
//                     one to its slot's integer counter: the result does not depend on the order, the grid or the trace variant.
//     k_ao_fold       per hit slot: the fragment of value 1 - occluded / N, the film fold, the pixel's RNG state s * M^(2N).
//   No path outlives its iteration, so every iteration is a full wave with no tail.  Each of k_ao_primary and k_ao_occlusion
//   exists for the small-scene path (flat scene in shared memory, traverseSmall) and for the BVH (traverseScene / Trav rounds).
#pragma once
#include "dev_wavefront.cuh"

namespace prb {
// hit list length of the running iteration: two counters, alternating per iteration (AOState::parity); k_ao_primary clears the
// one the previous k_ao_fold read
constexpr int CNT_AO_HITS = CNT_ACTIVE + 2;
static_assert(CNT_AO_HITS + 1 < CNT_NEE, "the AO hit counters overlap the shading queues");

struct AOState {
	uint64_t* rng;		  // per slot: RNG state after the camera draws of the running sample (hit slots)
	uint32_t* occluded;	  // per slot: occlusion rays of the running sample that hit something
	uint32_t* hits;		  // slots whose camera ray hit, in this iteration
	const uint64_t* jump; // jump[j] = M^(2j) mod 2^64 for j = 0 .. n (M: the pcg32_fast multiplier)
	uint32_t n;			  // occlusion rays per sample (prb_integrator::sample_count)
	uint32_t parity;	  // iteration & 1: which CNT_AO_HITS counter is in use
};

// the render of an integrator whose samples end at the first hit ('ao', 'vf') starts: iteration counters, and for a render from
// scratch the per-pixel sums (as k_init_slots does for 'direct')
PRB_DEV void beginFirstHitRender(const WFState& W, uint32_t slot)
{
	if (slot < W.nSlots) {
		const uint32_t pix = W.pixel[slot];
		W.iter[slot]		= W.firstIter;
		if (W.firstIter == 0) {
			W.sampleCount[pix] = 0;
			W.feedback[pix]	   = 0;
			if (W.varMean) {
#pragma unroll
				for (int k = 0; k < 3; ++k)
					W.varMean[3 * (size_t)pix + k] = W.varVar[3 * (size_t)pix + k] = 0.0f;
			}
			if (W.aov) {
#pragma unroll
				for (int k = 0; k < 10; ++k)
					W.aov[10 * (size_t)pix + k] = 0.0f;
			}
			if (W.aovExt) {
#pragma unroll
				for (int k = 0; k < (int)PRB_AOV_EXT; ++k)
					W.aovExt[PRB_AOV_EXT * (size_t)pix + k] = 0.0f;
			}
		}
	}
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		W.counters[CNT_END_ITER] = W.endIter;
		W.counters[CNT_WORK]	 = 0;
	}
}

__global__ void __launch_bounds__(128) k_ao_begin(WFState W, AOState A)
{
	const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
	beginFirstHitRender(W, slot);
	if (slot < W.nSlots)
		A.occluded[slot] = 0;
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		W.counters[CNT_AO_HITS]		= 0;
		W.counters[CNT_AO_HITS + 1] = 0;
	}
}

template <bool SMALL>
__global__ void __launch_bounds__(128) k_ao_primary(const __grid_constant__ DScene S, WFState W, AOState A)
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
	if (blockIdx.x == 0 && threadIdx.x == 0) {
		W.counters[CNT_AO_HITS + (A.parity ^ 1u)] = 0; // read by the previous k_ao_fold, which has finished (stream order)
		W.counters[CNT_WORK]					  = 0; // work counter of the next k_ao_occlusion
	}
	const bool live = it < endIter;
	if (!__any_sync(0xFFFFFFFFu, live)) // (warp-uniform; no barrier follows) the pixels of the warp have all their samples
		return;
	const bool groupMono = S.settings.spectral_mono || !S.settings.spectral_hero;
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
	bool hit	  = false;
	uint32_t sBg = 0;
	if (live) {
		W.iter[slot]		 = it + 1;
		const uint32_t flags = PRB_RAY_CAMERA | (cs.mono ? PRB_RAY_MONOCHROME : 0u);
		if (!found) { // handleZero: a zero fragment, which can only leave feedback bits
			++sBg;
			const Blob heroFactor = cs.mono ? heroOnly() : blob(1);
			const uint32_t fb	  = fragmentBitsZeroRadiance(S, heroFactor / (cs.wvlPDF * bsum(heroFactor)), blob(1), flags, groupMono);
			if (fb)
				W.feedback[pix] |= fb;
			foldSampleIntoFilm(W, pix, 0.0f, 0.0f, 0.0f, it + 1);
			W.rng[pix] = rnd.s;
		} else { // makeIP: RayStream::getRay re-normalises the camera ray on read, RayStream.cpp:167
			const V3 D = normalized(cs.dir);
			const V3 P = cs.origin + h.t * D;
			GeomPoint g;
			provideGeometryPointBody(S, h.entity, h.prim, h.u, h.v, P, g);
			addCameraVertex(W, pix, g, P, D, norm2(cs.origin - P)); // as 'direct' at path length 1
			W.vxP[slot]		   = make_float4(P.x, P.y, P.z, 0);
			W.vxN[slot]		   = make_float4(g.N.x, g.N.y, g.N.z, 0);
			W.vxNx[slot]	   = make_float4(g.Nx.x, g.Nx.y, g.Nx.z, 0);
			W.vxNy[slot]	   = make_float4(g.Ny.x, g.Ny.y, g.Ny.z, 0);
			W.wvl[slot]		   = tof4(cs.wvl);
			W.wvlPDF[slot]	   = tof4(cs.wvlPDF);
			W.flagsDepth[slot] = flags;
			A.rng[slot]		   = rnd.s;
			hit				   = true;
		}
	}
	warpAppend(W.counters + CNT_AO_HITS + A.parity, A.hits, hit, slot); // hit list
	{
		const uint32_t s = live ? 1u : 0u, e = hit ? 1u : 0u;
		const int which[6]	   = { ST_PIXEL_SAMPLE, ST_CAMERA_RAY, ST_PRIMARY, ST_ENTITY_HIT, ST_CAMERA_DEPTH, ST_BG_HIT };
		const uint32_t vals[6] = { s, s, s, e, e, sBg };
		statAddMany(W.stats, which, vals);
	}
}

// the occlusion ray of work item k, slot-major: the N rays of one hit point on consecutive lanes (profiles/r04_ao.txt)
PRB_DEV uint32_t aoItemRay(const WFState& W, const AOState& A, uint32_t k, V3& O, V3& D)
{
	const uint32_t slot = A.hits[k / A.n], j = k % A.n;
	Rng r{ A.rng[slot] * A.jump[j] };
	const float u2 = r.getFloat(); // cos_hemi(getFloat(), getFloat()) evaluated right to left, as the Lambert sampler draws
	const float u1 = r.getFloat();
	const float4 p = W.vxP[slot], n = W.vxN[slot], nx = W.vxNx[slot], ny = W.vxNy[slot];
	const V3 N = mk(n.x, n.y, n.z);
	D		   = fromTangentSpace(N, mk(nx.x, nx.y, nx.z), mk(ny.x, ny.y, ny.z), cos_hemi(u1, u2));
	// IntersectionPoint::nextRay (IntersectionPoint.h:116-124): the origin is pushed off the surface on the side of the ray
	O = safePosition(mk(p.x, p.y, p.z), D, dot(D, N) < 0 ? -N : N);
	return slot;
}

template <bool SMALL>
__global__ void __launch_bounds__(128) k_ao_occlusion(const __grid_constant__ DScene S, WFState W, AOState A)
{
	const uint32_t total = W.counters[CNT_AO_HITS + A.parity] * A.n; // the host keeps slots x n below 2^32
	if (SMALL) {
		__shared__ uint4 smallScene[SMALL ? SMALL_SCENE_U4 : 1];
		if (blockIdx.x * blockDim.x >= total)
			return;
		for (uint32_t i = threadIdx.x; i < S.nSmallU4; i += blockDim.x)
			smallScene[i] = __ldg(S.small + i);
		__syncthreads();
		// grid-stride over the items in whole warps (traverseSmall is warp-synchronous)
		const uint32_t lane = threadIdx.x & 31;
		for (uint32_t base = blockIdx.x * blockDim.x + (threadIdx.x - lane); base < total; base += gridDim.x * blockDim.x) {
			const uint32_t k = base + lane;
			const bool live	 = k < total;
			V3 O = mk(0, 0, 0), D = mk(0, 0, 1);
			uint32_t slot = 0;
			if (live)
				slot = aoItemRay(W, A, k, O, D);
			HitRec h;
			if (traverseSmall(smallScene, S.nSmallEnts, S.nSmallFaces, live, true, O, D, 0.0001f, PRB_INF, h) && live)
				atomicAdd(A.occluded + slot, 1u);
		}
	} else { // persistent Trav rounds, idle lanes refilled from the work counter (as the ray-stream kernels)
		Trav tr;
		uint2 stack[BVH_STACK_ALLOC];
		tr.idle();
		uint32_t slot = 0;
		bool active = false, pool = true;
		for (;;) {
			{
				const bool need	 = !active && pool;
				const uint32_t k = fetchWork(W.counters + CNT_WORK, need);
				if (need) {
					if (k < total) {
						V3 O, D;
						slot = aoItemRay(W, A, k, O, D);
						tr.begin(S, O, D, 0.0001f, PRB_INF, true, stack);
						active = true;
					} else {
						pool = false;
					}
				}
			}
			if (__ballot_sync(0xFFFFFFFFu, active) == 0)
				break;
			for (;;) {
				if (tr.round(S, active, stack)) {
					if (tr.hit())
						atomicAdd(A.occluded + slot, 1u);
					active = false;
				}
				const unsigned am = __ballot_sync(0xFFFFFFFFu, active);
				if (am == 0 || (__popc(am) < REFILL_LANES_STREAM && __any_sync(0xFFFFFFFFu, pool && !active)))
					break;
			}
		}
	}
}

__global__ void __launch_bounds__(128) k_ao_fold(const __grid_constant__ DScene S, WFState W, AOState A)
{
	const uint32_t i	 = blockIdx.x * blockDim.x + threadIdx.x;
	const uint32_t nHits = W.counters[CNT_AO_HITS + A.parity];
	if (blockIdx.x * blockDim.x >= nHits)
		return; // whole block past the end of the list
	uint32_t rays = 0;
	if (i < nHits) {
		const uint32_t slot	 = A.hits[i];
		const uint32_t pix	 = W.pixel[slot];
		const uint32_t flags = W.flagsDepth[slot];
		const float d		 = 1.0f - (float)A.occluded[slot] / (float)A.n;
		const Blob wvlPDF	 = blob4(W.wvlPDF[slot]);
		const Blob heroFactor = (flags & PRB_RAY_MONOCHROME) ? heroOnly() : blob(1);
		const bool groupMono  = S.settings.spectral_mono || !S.settings.spectral_hero;
		float xyz[3];
		const uint32_t fb = fragmentXYZ(S, heroFactor / (wvlPDF * bsum(heroFactor)), blob(1), blob(d), flags, groupMono, blob4(W.wvl[slot]), xyz);
		if (fb) // (a rejected fragment leaves xyz at zero)
			W.feedback[pix] |= fb;
		foldSampleIntoFilm(W, pix, xyz[0], xyz[1], xyz[2], W.iter[slot]);
		W.rng[pix]		 = A.rng[slot] * A.jump[A.n];
		A.occluded[slot] = 0;
		rays			 = A.n;
	}
	statAdd(W.stats, ST_SHADOW, rays);
}
} // namespace prb
