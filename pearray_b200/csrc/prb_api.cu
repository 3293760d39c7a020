// C-ABI implementation (include/prb200_abi.h) over the CUDA kernels.  sm_100a only; no CPU fallback: every
// entry point fails with PRB_ERR_NO_DEVICE / PRB_ERR_CUDA when no B200-class device is usable.
#include "dev_vf.cuh"

#include <dlfcn.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

using namespace prb;

// Staged shading (k_shade_geom / _nee / _scatter per material type) against the single k_shade: films are bit-identical, which
// one is faster depends on the scene (boltsandgears 164 -> 233 Msamples/s staged, cornellbox_glassy 51 -> 39), so a context
// MEASURES both on the first poll intervals of a render and keeps the faster (PRB_STAGED=0|1 pins the choice).

namespace {
thread_local std::string g_err;
prb_status fail(prb_status code, const std::string& msg)
{
	g_err = msg;
	return code;
}
#define CU(x)                                                                                                     \
	do {                                                                                                          \
		cudaError_t e_ = (x);                                                                                     \
		if (e_ != cudaSuccess)                                                                                    \
			return fail(PRB_ERR_CUDA, std::string(#x) + ": " + cudaGetErrorString(e_));                           \
	} while (0)

// a device buffer that frees itself; movable, not copyable
template <typename T>
struct DBuf {
	T* p	 = nullptr;
	size_t n = 0;
	DBuf() = default;
	DBuf(DBuf&& o) noexcept { *this = std::move(o); }
	DBuf& operator=(DBuf&& o) noexcept
	{
		std::swap(p, o.p);
		std::swap(n, o.n);
		return *this;
	}
	~DBuf() { release(); }
	cudaError_t alloc(size_t count)
	{
		if (count <= n && p)
			return cudaSuccess;
		release();
		n = count;
		if (count == 0)
			return cudaSuccess;
		return cudaMalloc(&p, count * sizeof(T));
	}
	cudaError_t upload(const T* h, size_t count, cudaStream_t s)
	{
		cudaError_t e = alloc(std::max<size_t>(count, 1));
		if (e != cudaSuccess || count == 0)
			return e;
		return cudaMemcpyAsync(p, h, count * sizeof(T), cudaMemcpyHostToDevice, s);
	}
	void release()
	{
		if (p)
			cudaFree(p);
		p = nullptr;
		n = 0;
	}
};

// one CUDA runtime handle (stream, event, graph exec, pinned block), passed to Destroy when the owner goes; movable, not copyable
template <typename H, auto Destroy>
struct Owned {
	H h = nullptr;
	Owned() = default;
	explicit Owned(H handle) : h(handle) {}
	Owned(Owned&& o) noexcept { std::swap(h, o.h); }
	~Owned() { reset(); }
	void reset()
	{
		if (h)
			Destroy(h);
		h = nullptr;
	}
	operator H() const { return h; }
};
using Event = Owned<cudaEvent_t, cudaEventDestroy>;

// an instantiated CUDA graph and the key naming everything its captured launches depend on
struct CachedGraph {
	Owned<cudaGraphExec_t, cudaGraphExecDestroy> exec;
	uint64_t key[7] = {};
	// re-captures what enqueue() launches on s unless the graph was captured for `k`
	template <class Enqueue>
	prb_status update(cudaStream_t s, const uint64_t (&k)[7], const Enqueue& enqueue)
	{
		if (exec && std::memcmp(k, key, sizeof(key)) == 0)
			return PRB_OK;
		exec.reset();
		cudaGraph_t graph = nullptr;
		cudaError_t be	  = cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal);
		if (be == cudaSuccess)
			enqueue();
		const cudaError_t ce = be == cudaSuccess ? cudaGetLastError() : be;
		const cudaError_t ee = be == cudaSuccess ? cudaStreamEndCapture(s, &graph) : be;
		if (ce != cudaSuccess || ee != cudaSuccess) {
			if (graph)
				cudaGraphDestroy(graph);
			return fail(PRB_ERR_CUDA, std::string("graph capture failed: ") + cudaGetErrorString(ce != cudaSuccess ? ce : ee));
		}
		const cudaError_t ie = cudaGraphInstantiate(&exec.h, graph, 0);
		cudaGraphDestroy(graph);
		if (ie != cudaSuccess) {
			exec.h = nullptr;
			return fail(PRB_ERR_CUDA, std::string("graph instantiation failed: ") + cudaGetErrorString(ie));
		}
		std::memcpy(key, k, sizeof(key));
		return PRB_OK;
	}
};
} // namespace

// Every device buffer and handle below frees itself.  Members go in reverse order of declaration, so the stream, declared
// first, outlives everything that was enqueued on it.
struct prb_ctx {
	int device = 0;
	Owned<cudaStream_t, cudaStreamDestroy> stream;
	Event evA, evB, evT0, evT1;
	~prb_ctx()
	{
		cudaSetDevice(device);
		if (stream)
			cudaStreamSynchronize(stream);
		prb_comm_destroy(this);
	}
	int smCount = 148;
	bool allLambert = false;	 // every material is PRB_MAT_DIFFUSE: k_shade with the Lambert code inline
	bool hasImageNodes = false;	 // some node is an image texture: no kernel with the Lambert code inline (leaf-only node evaluation)
	bool mixedMaterials = false; // the scene mixes material types: k_shade sorts larger windows (launchShade)
	int gridTrace = 148 * 4, gridTraceClosest = 148 * 4, gridTraceAny = 148 * 4; // persistent grids: SMs x resident blocks
	bool haveScene = false;
	DScene S{};
	// scene storage
	DBuf<prb_node> nodes;
	DBuf<prb_material> materials;
	DBuf<prb_emission> emissions;
	DBuf<prb_entity> entities;
	DBuf<uint32_t> entityMaterials, faceIndices, faceSlots, tlasRefs;
	DBuf<prb_mesh> meshes;
	DBuf<float> vertices, normals, uvs, lightCDF, pool, rrProb;
	DBuf<prb_light> lights;
	DBuf<uint4> bvhNodes;
	DBuf<float4> bvhTris;
	// film
	DBuf<uint64_t> rng;
	DBuf<float> filmMean, filmTmp, aov, aovExt, varMean, varVar; // varMean / varVar only with prb_settings.want_variance
	DBuf<uint32_t> sampleCount, feedback;
	DBuf<unsigned long long> stats;
	bool rngUploaded = false;
	uint32_t lastFirstIter = 0, lastEndIter = 0; // iteration range of the last prb_render_tiles call (sample-range film weights)
	// multi-GPU film combine
	void* ncclComm = nullptr;
	int commRank = 0, commWorld = 1;
	DBuf<float> reduceF;	 // FILM_PACK floats per pixel
	DBuf<uint32_t> reduceU;	 // spread feedback bits
	float lastReduceMs = 0;
	// wavefront
	DBuf<uint32_t> pixel, iter, flagsDepth, slotState, counters, regenList, activeList, neeList, scatterList;
	DBuf<float4> rayO, rayD, wvl, thr, pathPDF, prevPDF, wvlPDF, lastPos, shO, shD, shXYZ, iterXYZ, prevAcc, vxP, vxN, vxNx, vxNy, vxD;
	bool staged = false;	   // k_shade_geom -> k_shade_nee / k_shade_scatter per material type instead of k_shade
	bool stagedAuto = false;   // not pinned: decided by measurement (tuneStep / tuneMs) during the first render of the scene
	int tuneStep = 0;		   // poll intervals measured so far (modes 0,1,1,0: cancels the drift of the falling path count)
	float tuneMs[2] = { 0, 0 };
	uint8_t queueOfType[SHADE_QUEUES];	   // material type -> queue index, 0xFF when the scene has no material of the type
	bool queueWantsNEE[SHADE_QUEUES] = {}; // some material of the queue's type has a non-delta lobe
	uint32_t nQueues = 0, nNeeQueues = 0;
	uint32_t launchesPerIteration(bool stagedMode) const { return (stagedMode ? 3 + nQueues + nNeeQueues : 3) - (regenInTrace() ? 1 : 0) + (persistentTrace ? 1 : 0); }
	bool regenInTrace() const { return smallScene && !persistentTrace; }
	// all-Lambert small scenes: k_trace_small lists the slots whose path goes on, k_shade walks the list (PRB_COMPACT_SMALL=0 / 1
	// overrides).  Dense warps pay once k_shade is throughput bound, i.e. from about two waves of its blocks (4 x 128 slots per SM):
	// cornellbox 500 x 500: 373.8 -> 384.0 Msamples/s; the 256 x 256 evaluation scene, one wave, loses the extra dependent load
	// (249.6 -> 244.9)
	bool compactSmall() const
	{
		if (!regenInTrace() || !allLambert)
			return false;
		if (const char* e = std::getenv("PRB_COMPACT_SMALL"))
			return e[0] != '0';
		return nSlots >= (size_t)smCount * 4 * 128 * 2;
	} // k_trace_small regenerates ended paths itself: no k_regen launch
	DBuf<uint4> hit;
	DBuf<float> hitT;
	// light path expression channels (scenes with prb_scene_desc::n_lpe > 0)
	DBuf<uint8_t> lpeTables;
	DBuf<uint2> lpeState;
	DBuf<float4> lpeAcc, lpePrev;
	DBuf<float> lpeFilm; // n_lpe films of npix * 3 floats
	std::vector<prb_tile> cachedTiles;
	uint32_t nSlots = 0;
	Owned<uint32_t*, cudaFreeHost> hostCounters; // pinned
	// generic scratch for the host-pointer entry points
	DBuf<float> scratchF;
	DBuf<uint32_t> scratchU;
	DBuf<uint8_t> scratchB;
	DBuf<prb_material_query> scratchQ;
	DBuf<prb_material_result> scratchR;
	// bookkeeping
	uint64_t kernelLaunches = 0, wavefrontIterations = 0;
	float lastMs = 0;
	// the wavefront graph (ITERS_PER_GRAPH x k_trace, k_shade, k_regen) is instantiated once and replayed by every
	// prb_render_tiles call until something baked into its kernel parameters changes (scene, slot buffers, variant)
	CachedGraph directGraph[2]; // [staged]
	uint64_t stateVersion = 1; // bumped whenever the scene or the slot buffers change
	bool wantAOV = true;
	bool persistentTrace = true; // k_trace (persistent threads) vs k_trace_static, chosen per scene in prb_upload_scene
	bool smallScene = false;	 // k_trace_small: a tiny scene traced from shared memory, no BVH
	DBuf<uint4> small;
	// per-stage profiling (prb_set_profiling)
	bool profiling = false;
	std::vector<Event> profEvents; // pairs
	float stageMs[PRB_STAGE__COUNT] = {};
	uint64_t stageLaunches[PRB_STAGE__COUNT] = {};
	// the integrator prb_render_tiles runs (prb_set_integrator; prb_upload_scene resets it to 'direct')
	prb_integrator integrator{ PRB_INTEGRATOR_DIRECT, 0 };
	// 'ao': per-slot state of the running sample, the hit list, the jump-ahead table
	DBuf<uint64_t> aoRng, aoJump;
	DBuf<uint32_t> aoOccluded, aoHits;
	int gridAOSmall = 148 * 4, gridAO = 148 * 4; // persistent k_ao_occlusion grids
	// 'ao' and 'vf': the graph of ITERS_PER_GRAPH iterations (renderFirstHit) and what it was captured for
	CachedGraph firstHitGraph;
};

// grows the pool of profiling events to at least n
static prb_status reserveProfEvents(prb_ctx* c, size_t n)
{
	while (c->profEvents.size() < n) {
		cudaEvent_t ev;
		CU(cudaEventCreate(&ev));
		c->profEvents.emplace_back(ev);
	}
	return PRB_OK;
}

template <int KIND>
static void launchStageKernels(prb_ctx* c, const WFState& W, uint32_t queue, cudaStream_t s)
{
	const int grid = (int)((c->nSlots + 127) / 128);
	if (c->S.nLPE) {
		if (c->queueWantsNEE[queue]) // (a queue of delta-only materials never does NEE)
			k_shade_nee<KIND, true><<<grid, 128, 0, s>>>(c->S, W, queue);
		k_shade_scatter<KIND, true><<<grid, 128, 0, s>>>(c->S, W, queue);
	} else {
		if (c->queueWantsNEE[queue])
			k_shade_nee<KIND, false><<<grid, 128, 0, s>>>(c->S, W, queue);
		k_shade_scatter<KIND, false><<<grid, 128, 0, s>>>(c->S, W, queue);
	}
}

extern "C" {
const char* prb_last_error(void) { return g_err.c_str(); }

int prb_device_count(void)
{
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess)
		return 0;
	return n;
}

prb_status prb_create(int device, prb_ctx** out)
{
	if (!out)
		return fail(PRB_ERR_INVALID_ARG, "out == NULL");
	*out  = nullptr;
	int n = 0;
	if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0)
		return fail(PRB_ERR_NO_DEVICE, "no CUDA device available (the path has no CPU fallback)");
	if (device < 0 || device >= n)
		return fail(PRB_ERR_INVALID_ARG, "invalid device index");
	CU(cudaSetDevice(device));
	cudaDeviceProp prop;
	CU(cudaGetDeviceProperties(&prop, device));
	if (prop.major < 10)
		return fail(PRB_ERR_NO_DEVICE, std::string("device '") + prop.name + "' is not sm_100-class; this library is built for sm_100a only");
	auto* c		= new prb_ctx();
	c->device	= device;
	c->smCount	= prop.multiProcessorCount;
	cudaError_t e = cudaStreamCreateWithFlags(&c->stream.h, cudaStreamNonBlocking);
	for (Event* ev : { &c->evA, &c->evB, &c->evT0, &c->evT1 })
		if (e == cudaSuccess)
			e = cudaEventCreate(&ev->h);
	if (e == cudaSuccess)
		e = cudaMallocHost(&c->hostCounters.h, CNT__COUNT * sizeof(uint32_t));
	if (e == cudaSuccess)
		e = c->stats.alloc(ST__COUNT);
	if (e == cudaSuccess)
		e = cudaMemsetAsync(c->stats.p, 0, ST__COUNT * sizeof(unsigned long long), c->stream);
	if (e == cudaSuccess) {
		// persistent-thread kernels: one grid that exactly fills the machine (SM count x resident blocks per SM)
		int nb = 0;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace, 128, 0) == cudaSuccess && nb > 0)
			c->gridTrace = c->smCount * nb;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace_closest, 128, 0) == cudaSuccess && nb > 0)
			c->gridTraceClosest = c->smCount * nb;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_trace_any, 128, 0) == cudaSuccess && nb > 0)
			c->gridTraceAny = c->smCount * nb;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_ao_occlusion<true>, 128, 0) == cudaSuccess && nb > 0)
			c->gridAOSmall = c->smCount * nb;
		if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, k_ao_occlusion<false>, 128, 0) == cudaSuccess && nb > 0)
			c->gridAO = c->smCount * nb;
	}
	if (e != cudaSuccess) {
		delete c;
		return fail(PRB_ERR_CUDA, std::string("context set-up failed: ") + cudaGetErrorString(e));
	}
	*out = c;
	return PRB_OK;
}

void prb_destroy(prb_ctx* c) { delete c; }

// number of BVH8 levels below (and including) `root`; 0 when an index is out of range or the tree is deeper than `limit`
static uint32_t bvhLevels(const prb_scene_desc* d, uint32_t root, uint32_t limit)
{
	struct Item {
		uint32_t node, level;
	};
	std::vector<Item> todo{ { root, 1 } };
	uint32_t deepest = 0;
	while (!todo.empty()) {
		const Item it = todo.back();
		todo.pop_back();
		if (it.node >= d->n_bvh_nodes || it.level > limit)
			return 0;
		deepest					= std::max(deepest, it.level);
		const prb_bvh8_node& n = d->bvh_nodes[it.node];
		for (int i = 0; i < 8; ++i)
			if (n.meta[i] != 0xFF && (n.meta[i] & 0x80))
				todo.push_back({ n.child_base + (n.meta[i] & 0x7Fu), it.level + 1 });
	}
	return deepest;
}

prb_status prb_upload_scene(prb_ctx* c, const prb_scene_desc* d)
{
	if (!c || !d)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (d->abi_version != PRB_ABI_VERSION)
		return fail(PRB_ERR_INVALID_ARG, "scene descriptor ABI version mismatch");
	{
		// The traversal stack holds BVH_STACK groups per ray.  A node visit parks at most two groups (the unvisited hit
		// children and the hit leaf primitives), entering a BLAS three (both TLAS groups and the exit marker), so a scene
		// needs 2 x TLAS levels + 3 + 2 x deepest BLAS levels entries; a deeper BVH would silently drop subtrees, so it is
		// rejected here instead.
		const uint32_t limit = BVH_STACK;
		const uint32_t tlas	 = bvhLevels(d, d->tlas_root, limit);
		uint32_t blas		 = 0;
		bool ok				 = tlas != 0;
		std::vector<uint32_t> seen;
		for (uint32_t i = 0; ok && i < d->n_entities; ++i) {
			const uint32_t r = d->entities[i].blas_root;
			if (d->entities[i].type == PRB_ENTITY_SPHERE || r == PRB_INVALID_ID || std::find(seen.begin(), seen.end(), r) != seen.end())
				continue;
			seen.push_back(r);
			const uint32_t l = bvhLevels(d, r, limit);
			ok				 = l != 0;
			blas			 = std::max(blas, l);
		}
		if (!ok || 2 * tlas + 3 + 2 * blas > (uint32_t)BVH_STACK)
			return fail(PRB_ERR_UNSUPPORTED, "BVH too deep for the " + std::to_string(BVH_STACK) + "-entry traversal stack (or a node index is out of range): TLAS " +
												 std::to_string(tlas) + " levels, deepest BLAS " + std::to_string(blas) + " levels");
	}
	static_assert(sizeof(prb_bvh8_node) == 80, "node must be 80 bytes");
	static_assert(sizeof(prb_bvh_tri) == 48, "triangle must be 48 bytes");
	CU(cudaSetDevice(c->device));
	cudaStream_t s = c->stream;
	CU(c->nodes.upload(d->nodes, d->n_nodes, s));
	CU(c->materials.upload(d->materials, d->n_materials, s));
	CU(c->emissions.upload(d->emissions, d->n_emissions, s));
	CU(c->entities.upload(d->entities, d->n_entities, s));
	CU(c->entityMaterials.upload(d->entity_materials, d->n_entity_materials, s));
	CU(c->meshes.upload(d->meshes, d->n_meshes, s));
	CU(c->vertices.upload(d->vertices, (size_t)d->n_vertices * 3, s));
	CU(c->normals.upload(d->normals, (size_t)d->n_vertices * 3, s));
	CU(c->uvs.upload(d->uvs, (size_t)d->n_vertices * 2, s));
	CU(c->faceIndices.upload(d->face_indices, (size_t)d->n_faces * 4, s));
	CU(c->faceSlots.upload(d->face_slots, d->n_faces, s));
	CU(c->lights.upload(d->lights, d->n_lights, s));
	CU(c->lightCDF.upload(d->light_cdf, (size_t)d->n_lights + 1, s));
	CU(c->bvhNodes.upload(reinterpret_cast<const uint4*>(d->bvh_nodes), (size_t)d->n_bvh_nodes * 5, s));
	CU(c->bvhTris.upload(reinterpret_cast<const float4*>(d->bvh_tris), (size_t)d->n_bvh_tris * 3, s));
	CU(c->tlasRefs.upload(d->tlas_refs, d->n_tlas_refs, s));
	CU(c->pool.upload(d->pool, d->n_pool, s));
	for (uint32_t i = 0; i < d->n_nodes; ++i) {
		const prb_node& n = d->nodes[i];
		if (n.type != PRB_NODE_IMAGE)
			continue;
		const uint64_t w = n.b & 0xFFFFu, h = n.b >> 16, res = d->upsampler_res;
		if (w == 0 || h == 0 || (uint64_t)n.a + w * h * 3 > d->n_pool)
			return fail(PRB_ERR_INVALID_ARG, "image node " + std::to_string(i) + ": texels outside the pool");
		if (res < 2 || (uint64_t)d->upsampler_offset + res + 9 * res * res * res > d->n_pool)
			return fail(PRB_ERR_INVALID_ARG, "image node " + std::to_string(i) + ": the scene carries no spectral upsampler table");
	}
	if (d->n_lpe > PRB_MAX_LPE)
		return fail(PRB_ERR_INVALID_ARG, "more than PRB_MAX_LPE light path expressions");
	for (uint32_t k = 0; k < d->n_lpe; ++k) {
		const prb_lpe& l = d->lpe[k];
		if (l.n_states == 0 || l.n_states > 255 || l.start_state >= l.n_states || !d->lpe_tables ||
			(uint64_t)l.next_offset + (uint64_t)l.n_states * PRB_LPE_SYMBOLS > d->n_lpe_bytes || (uint64_t)l.final_offset + l.n_states > d->n_lpe_bytes)
			return fail(PRB_ERR_INVALID_ARG, "light path expression " + std::to_string(k) + ": table out of range");
		for (uint32_t i = 0; i < l.n_states * PRB_LPE_SYMBOLS; ++i) {
			const uint8_t n = d->lpe_tables[l.next_offset + i];
			if (n != PRB_LPE_REJECT && n >= l.n_states)
				return fail(PRB_ERR_INVALID_ARG, "light path expression " + std::to_string(k) + ": transition to a state that does not exist");
		}
	}
	c->S.nLPE	   = d->n_lpe;
	c->S.lpeTables = nullptr;
	std::memcpy(c->S.lpe, d->lpe, sizeof(c->S.lpe));
	if (d->n_lpe) {
		CU(c->lpeTables.upload(d->lpe_tables, d->n_lpe_bytes, s));
		c->S.lpeTables = c->lpeTables.p;
	}
	// RussianRoulette::probability table (vcm/RussianRoulette.h:22-34): min(1, pow(0.9f, len - soft)) evaluated in
	// double and rounded to float exactly like std::pow(float, size_t) does on the host
	const uint32_t soft = d->settings.soft_max_ray_depth;
	const uint32_t nrr	= std::max(d->settings.max_ray_depth, soft) + 5;
	std::vector<float> rr(nrr, 1.0f);
	for (uint32_t len = 0; len < nrr; ++len)
		if (len >= soft) {
			const float p = std::min<float>(1.0f, (float)std::pow((double)0.9f, (double)(len - soft)));
			rr[len]		  = p <= 1e-4f ? 0.0f : p;
		}
	CU(c->rrProb.upload(rr.data(), rr.size(), s));
	const size_t npix = (size_t)d->settings.film_width * d->settings.film_height;
	CU(c->rng.alloc(npix));
	CU(c->filmMean.alloc(npix * 3));
	CU(c->filmTmp.alloc(npix * 4));
	CU(c->sampleCount.alloc(npix));
	CU(c->aov.alloc(npix * 10));
	if (d->settings.want_aov_ext) {
		CU(c->aovExt.alloc(npix * PRB_AOV_EXT));
		CU(cudaMemsetAsync(c->aovExt.p, 0, npix * PRB_AOV_EXT * sizeof(float), s));
	} else {
		c->aovExt.release();
	}
	CU(c->feedback.alloc(npix));
	CU(cudaMemsetAsync(c->feedback.p, 0, npix * sizeof(uint32_t), s));
	if (d->n_lpe) {
		CU(c->lpeFilm.alloc(npix * 3 * d->n_lpe));
		CU(cudaMemsetAsync(c->lpeFilm.p, 0, npix * 3 * d->n_lpe * sizeof(float), s));
	} else {
		c->lpeFilm.release();
	}
	if (d->settings.want_variance) {
		CU(c->varMean.alloc(npix * 3));
		CU(c->varVar.alloc(npix * 3));
		CU(cudaMemsetAsync(c->varMean.p, 0, npix * 3 * sizeof(float), s));
		CU(cudaMemsetAsync(c->varVar.p, 0, npix * 3 * sizeof(float), s));
	} else {
		c->varMean.release();
		c->varVar.release();
	}
	CU(cudaMemsetAsync(c->filmMean.p, 0, npix * 3 * sizeof(float), s));
	CU(cudaMemsetAsync(c->sampleCount.p, 0, npix * sizeof(uint32_t), s));
	CU(cudaMemsetAsync(c->aov.p, 0, npix * 10 * sizeof(float), s));
	CU(cudaMemsetAsync(c->rng.p, 0, npix * sizeof(uint64_t), s));
	DScene& S		  = c->S;
	S.settings		  = d->settings;
	S.camera		  = d->camera;
	S.aa			  = d->aa_sampler;
	S.lens			  = d->lens_sampler;
	S.time			  = d->time_sampler;
	S.mapper		  = d->pixel_mapper;
	S.nodes			  = c->nodes.p;
	S.materials		  = c->materials.p;
	S.emissions		  = c->emissions.p;
	S.entities		  = c->entities.p;
	S.entityMaterials = c->entityMaterials.p;
	S.meshes		  = c->meshes.p;
	S.vertices		  = c->vertices.p;
	S.normals		  = c->normals.p;
	S.uvs			  = c->uvs.p;
	S.faceIndices	  = c->faceIndices.p;
	S.faceSlots		  = c->faceSlots.p;
	S.lights		  = c->lights.p;
	S.lightCDF		  = c->lightCDF.p;
	S.bvhNodes		  = c->bvhNodes.p;
	S.bvhTris		  = c->bvhTris.p;
	S.tlasRefs		  = c->tlasRefs.p;
	S.pool			  = c->pool.p;
	S.rrProb		  = c->rrProb.p;
	S.rrCount		  = nrr;
	S.nMaterials	  = d->n_materials;
	S.nEmissions	  = d->n_emissions;
	S.nEntities		  = d->n_entities;
	S.nLights		  = d->n_lights;
	S.nMeshes		  = d->n_meshes;
	S.tlasRoot		  = d->tlas_root;
	S.cieOffset		  = d->cie_offset;
	S.upsamplerOffset = d->upsampler_offset;
	S.upsamplerRes	  = d->upsampler_res;
	c->mixedMaterials = false;
	c->allLambert	  = d->n_materials > 0 && d->materials[0].type == PRB_MAT_DIFFUSE;
	c->hasImageNodes = false;
	for (uint32_t i = 0; i < d->n_nodes; ++i) // the kernels with the Lambert code inline evaluate nodes without the image-texture path
		if (d->nodes[i].type == PRB_NODE_IMAGE)
			c->hasImageNodes = true;
	if (c->hasImageNodes)
		c->allLambert = false;
	for (uint32_t i = 1; i < d->n_materials; ++i)
		if (d->materials[i].type != d->materials[0].type)
			c->mixedMaterials = true;
	S.hasCombined	  = 0;
	for (uint32_t i = 0; i < d->n_materials; ++i)
		if (d->materials[i].type == PRB_MAT_BLEND || d->materials[i].type == PRB_MAT_ADD)
			S.hasCombined = 1;
	S.hasInfLight	  = 0;
	for (uint32_t i = 0; i < d->n_lights; ++i)
		if (d->lights[i].type != PRB_LIGHT_AREA)
			S.hasInfLight = 1;
	CU(cudaStreamSynchronize(s));
	// trace-kernel variant: persistent threads pay off once rays take many traversal steps (measured: 2x on the 10 M
	// triangle soup, 0.7x on the 32-triangle Cornell box, 1.0x on the 6 k-triangle bolts scene, 1.09x on complex.prc with 53 k); PRB_TRACE_MODE=static|persistent overrides the heuristic
	c->persistentTrace = d->n_bvh_tris > 32768;
	if (const char* m = std::getenv("PRB_TRACE_MODE")) {
		if (std::strcmp(m, "static") == 0)
			c->persistentTrace = false;
		else if (std::strcmp(m, "persistent") == 0)
			c->persistentTrace = true;
	}
	// tiny scenes: flat entity / triangle list for the BVH-free trace kernel (traverseSmall)
	c->smallScene	= false;
	c->S.small		= nullptr;
	c->S.nSmallEnts = c->S.nSmallFaces = c->S.nSmallU4 = 0;
	if (!c->persistentTrace && d->n_bvh_tris <= SMALL_MAX_TRIS && d->n_entities <= SMALL_MAX_ENTS && d->n_entities > 0) {
		std::vector<uint4> blob(4 * (size_t)d->n_entities), tris;
		std::vector<float4> boxes; // per face: lo (w: first triangle), hi (w: triangle count)
		bool ok = true;
		for (uint32_t e = 0; e < d->n_entities && ok; ++e) {
			const prb_entity& en = d->entities[e];
			uint4 h				 = make_uint4(en.type, e, 0, 0);
			float rows[12]		 = {};
			if (en.type == PRB_ENTITY_SPHERE) {
				rows[0] = en.geo[0], rows[1] = en.geo[1], rows[2] = en.geo[2], rows[3] = en.geo[3];
			} else {
				std::memcpy(rows, en.world_to_local, sizeof(rows));
				// every triangle below the BLAS root
				std::vector<prb_bvh_tri> own;
				std::vector<uint32_t> todo{ en.blas_root };
				while (!todo.empty() && ok) {
					const uint32_t ni = todo.back();
					todo.pop_back();
					if (ni >= d->n_bvh_nodes) {
						ok = false;
						break;
					}
					const prb_bvh8_node& n = d->bvh_nodes[ni];
					for (int i = 0; i < 8; ++i) {
						if (n.meta[i] == 0xFF)
							continue;
						if (n.meta[i] & 0x80) {
							todo.push_back(n.child_base + (n.meta[i] & 0x7Fu));
						} else {
							const uint32_t count = ((n.meta[i] >> 5) & 3u) + 1, first = n.prim_base + (n.meta[i] & 0x1Fu);
							for (uint32_t k = 0; k < count; ++k) {
								if (first + k >= d->n_bvh_tris) {
									ok = false;
									break;
								}
								own.push_back(d->bvh_tris[first + k]);
							}
						}
					}
				}
				// faces: two triangles share one box when the union of their world-space boxes is hardly larger than the larger
				// of the two -- the halves of a quad, or the two triangles a modeller split a planar rectangle into (the walls
				// of the Cornell boxes); greedy, best partner first
				auto worldBox = [&](const prb_bvh_tri& bt, double lo[3], double hi[3]) {
					const float* vtx[3] = { bt.v0, bt.v1, bt.v2 };
					for (int a = 0; a < 3; ++a)
						lo[a] = 1e300, hi[a] = -1e300;
					for (int j = 0; j < 3; ++j)
						for (int a = 0; a < 3; ++a) {
							double w = vtx[j][a];
							if (en.type == PRB_ENTITY_MESH) {
								const float* m = en.local_to_world + 4 * a;
								w			   = (double)m[0] * vtx[j][0] + (double)m[1] * vtx[j][1] + (double)m[2] * vtx[j][2] + (double)m[3];
							}
							lo[a] = std::min(lo[a], w);
							hi[a] = std::max(hi[a], w);
						}
				};
				auto halfArea = [](const double lo[3], const double hi[3]) {
					const double x = hi[0] - lo[0], y = hi[1] - lo[1], z = hi[2] - lo[2];
					return x * y + y * z + z * x + 1e-3 * (x + y + z) * (x + y + z); // the second term orders flat (zero-area) boxes by extent
				};
				std::vector<prb_bvh_tri> paired;
				std::vector<char> used(own.size(), 0);
				std::vector<uint32_t> faceCount;
				for (size_t i = 0; i < own.size(); ++i) {
					if (used[i])
						continue;
					used[i] = 1;
					double li[3], hi_[3];
					worldBox(own[i], li, hi_);
					size_t bestJ	 = own.size();
					double bestRatio = 1.1;
					for (size_t j = i + 1; j < own.size(); ++j) {
						if (used[j])
							continue;
						double lj[3], hj[3], lu[3], hu[3];
						worldBox(own[j], lj, hj);
						for (int a = 0; a < 3; ++a)
							lu[a] = std::min(li[a], lj[a]), hu[a] = std::max(hi_[a], hj[a]);
						const double ratio = halfArea(lu, hu) / std::max(std::max(halfArea(li, hi_), halfArea(lj, hj)), 1e-300);
						if (ratio < bestRatio)
							bestRatio = ratio, bestJ = j;
					}
					paired.push_back(own[i]);
					faceCount.push_back(1);
					if (bestJ < own.size()) {
						used[bestJ] = 1;
						paired.push_back(own[bestJ]);
						faceCount.back() = 2;
					}
				}
				own.swap(paired);
				size_t face = 0;
				for (size_t i = 0; i < own.size(); ++face) {
					const size_t n = faceCount[face];
					// padded world-space box (traverseSmall, phase 1): mesh triangles are stored in the instance's local space, planes in world space
					double lo[3] = { 1e300, 1e300, 1e300 }, hi[3] = { -1e300, -1e300, -1e300 }, mag = 0;
					const uint32_t firstTri = (uint32_t)(tris.size() / 3);
					for (size_t k = i; k < i + n; ++k) {
						const prb_bvh_tri& bt = own[k];
						const uint4* t		  = reinterpret_cast<const uint4*>(&bt);
						tris.insert(tris.end(), t, t + 3);
						tris.back().w = e; // index of the entity header (traverseSmall, phase 2)
						const float* vtx[3] = { bt.v0, bt.v1, bt.v2 };
						for (int j = 0; j < 3; ++j)
							for (int a = 0; a < 3; ++a) {
								double w = vtx[j][a];
								if (en.type == PRB_ENTITY_MESH) {
									const float* m = en.local_to_world + 4 * a;
									w			   = (double)m[0] * vtx[j][0] + (double)m[1] * vtx[j][1] + (double)m[2] * vtx[j][2] + (double)m[3];
								}
								lo[a] = std::min(lo[a], w);
								hi[a] = std::max(hi[a], w);
								mag	  = std::max(mag, std::fabs(w));
							}
					}
					const double pad = std::max(8e-6 * mag, 1e-30);
					float4 blo, bhi;
					blo.x = std::nextafterf((float)(lo[0] - pad), -INFINITY), blo.y = std::nextafterf((float)(lo[1] - pad), -INFINITY),
					blo.z = std::nextafterf((float)(lo[2] - pad), -INFINITY);
					bhi.x = std::nextafterf((float)(hi[0] + pad), INFINITY), bhi.y = std::nextafterf((float)(hi[1] + pad), INFINITY),
					bhi.z = std::nextafterf((float)(hi[2] + pad), INFINITY);
					uint32_t cnt = (uint32_t)n;
					std::memcpy(&blo.w, &firstTri, 4);
					std::memcpy(&bhi.w, &cnt, 4);
					boxes.push_back(blo);
					boxes.push_back(bhi);
					i += n;
				}
			}
			blob[4 * e] = h;
			std::memcpy(&blob[4 * e + 1], rows, sizeof(rows));
		}
		const size_t nSmallFaces = boxes.size() / 2;
		if (ok && tris.size() / 3 <= SMALL_MAX_TRIS) {
			while (boxes.size() % 16) // the box loop of traverseSmall runs in groups of 8 (bits past the last face are masked off)
				boxes.push_back(make_float4(0, 0, 0, 0));
			const uint4* bx = reinterpret_cast<const uint4*>(boxes.data());
			blob.insert(blob.end(), bx, bx + boxes.size());
			blob.insert(blob.end(), tris.begin(), tris.end());
			CU(c->small.upload(blob.data(), blob.size(), s));
			CU(cudaStreamSynchronize(s));
			c->S.small		 = c->small.p;
			c->S.nSmallEnts	 = d->n_entities;
			c->S.nSmallFaces = (uint32_t)nSmallFaces;
			c->S.nSmallU4	 = (uint32_t)blob.size();
			c->smallScene	 = true;
		}
	}
	if (const char* m = std::getenv("PRB_TRACE_MODE"))
		if (std::strcmp(m, "bvh") == 0)
			c->smallScene = false;
	// staged shading pays off where material types mix (one compact kernel per type instead of one 400 KB kernel that is
	// instruction-fetch bound); an all-Lambert scene is served best by the single inlined k_shade (measured: C2 272 vs 226 M)
	c->staged	  = false;
	c->stagedAuto = !c->allLambert;
	c->tuneStep	  = 0;
	c->tuneMs[0] = c->tuneMs[1] = 0;
	if (const char* m = std::getenv("PRB_STAGED")) {
		c->staged	  = std::atoi(m) != 0;
		c->stagedAuto = false;
	}
	if (d->n_lpe) { // the light path expression channels are accumulated by the staged kernels only
		c->staged	  = true;
		c->stagedAuto = false;
	}
	std::memset(c->queueOfType, 0xFF, sizeof(c->queueOfType));
	std::memset(c->queueWantsNEE, 0, sizeof(c->queueWantsNEE));
	c->nQueues = 0;
	for (uint32_t i = 0; i < d->n_materials; ++i) {
		const uint32_t t = std::min<uint32_t>(d->materials[i].type, SHADE_QUEUES - 1);
		if (c->queueOfType[t] == 0xFF)
			c->queueOfType[t] = (uint8_t)c->nQueues++;
		if (!(d->materials[i].flags & PRB_MATF_ONLY_DELTA))
			c->queueWantsNEE[c->queueOfType[t]] = true;
	}
	c->nNeeQueues = 0;
	for (uint32_t q = 0; q < c->nQueues; ++q)
		c->nNeeQueues += c->queueWantsNEE[q] ? 1u : 0u;
	c->haveScene   = true;
	c->integrator  = prb_integrator{ PRB_INTEGRATOR_DIRECT, 0 };
	c->rngUploaded = false; // the RNG map was zeroed above: state 0 of the pcg32_fast MCG stays 0 forever
	c->cachedTiles.clear();
	c->nSlots = 0;
	c->stateVersion++;
	return PRB_OK;
}

prb_status prb_upload_rng(prb_ctx* c, const uint64_t* states, size_t n)
{
	if (!c || !states)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n != (size_t)c->S.settings.film_width * c->S.settings.film_height)
		return fail(PRB_ERR_INVALID_ARG, "rng state count must be film_width*film_height");
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(c->rng.p, states, n * sizeof(uint64_t), cudaMemcpyHostToDevice, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	c->rngUploaded = true;
	return PRB_OK;
}
prb_status prb_download_rng(prb_ctx* c, uint64_t* states, size_t n)
{
	if (!c || !states)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n != (size_t)c->S.settings.film_width * c->S.settings.film_height)
		return fail(PRB_ERR_INVALID_ARG, "rng state count must be film_width*film_height");
	CU(cudaSetDevice(c->device));
	CU(cudaMemcpyAsync(states, c->rng.p, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}

prb_status prb_film_clear(prb_ctx* c)
{
	if (!c || !c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	CU(cudaMemsetAsync(c->filmMean.p, 0, npix * 3 * sizeof(float), c->stream));
	CU(cudaMemsetAsync(c->sampleCount.p, 0, npix * sizeof(uint32_t), c->stream));
	CU(cudaMemsetAsync(c->aov.p, 0, npix * 10 * sizeof(float), c->stream));
	if (c->aovExt.p)
		CU(cudaMemsetAsync(c->aovExt.p, 0, npix * PRB_AOV_EXT * sizeof(float), c->stream));
	CU(cudaMemsetAsync(c->feedback.p, 0, npix * sizeof(uint32_t), c->stream));
	if (c->varMean.p) {
		CU(cudaMemsetAsync(c->varMean.p, 0, npix * 3 * sizeof(float), c->stream));
		CU(cudaMemsetAsync(c->varVar.p, 0, npix * 3 * sizeof(float), c->stream));
	}
	if (c->lpeFilm.p)
		CU(cudaMemsetAsync(c->lpeFilm.p, 0, npix * 3 * c->S.nLPE * sizeof(float), c->stream));
	return PRB_OK;
}

static prb_status setupSlots(prb_ctx* c, const prb_tile* tiles, size_t n_tiles)
{
	const bool same = c->cachedTiles.size() == n_tiles && (n_tiles == 0 || std::memcmp(c->cachedTiles.data(), tiles, n_tiles * sizeof(prb_tile)) == 0);
	if (same && c->nSlots > 0)
		return PRB_OK;
	const uint32_t W = c->S.settings.film_width, H = c->S.settings.film_height;
	std::vector<uint32_t> pix;
	std::vector<uint8_t> owned((size_t)W * H, 0); // slot == pixel: a pixel listed twice would race on its RNG state and film cell
	for (size_t t = 0; t < n_tiles; ++t) {
		if (tiles[t].ex > W || tiles[t].ey > H || tiles[t].sx >= tiles[t].ex || tiles[t].sy >= tiles[t].ey)
			return fail(PRB_ERR_INVALID_ARG, "tile outside the film");
		for (uint32_t y = tiles[t].sy; y < tiles[t].ey; ++y)
			for (uint32_t x = tiles[t].sx; x < tiles[t].ex; ++x) {
				if (owned[(size_t)y * W + x])
					return fail(PRB_ERR_INVALID_ARG, "tiles overlap: a film pixel may be listed only once per call");
				owned[(size_t)y * W + x] = 1;
				pix.push_back(y * W + x);
			}
	}
	const size_t n = pix.size();
	CU(c->pixel.upload(pix.data(), n, c->stream));
	CU(c->iter.alloc(n));
	CU(c->flagsDepth.alloc(n));
	CU(c->slotState.alloc(n));
	CU(c->regenList.alloc(n));
	CU(c->activeList.alloc(n));
	if (c->staged || c->stagedAuto) { // one queue per material type of the scene
		CU(c->neeList.alloc(n * std::max<size_t>(c->nQueues, 1)));
		CU(c->scatterList.alloc(n * std::max<size_t>(c->nQueues, 1)));
	}
	CU(c->counters.alloc(CNT__COUNT));
	DBuf<float4>* f4[] = { &c->rayO, &c->rayD, &c->wvl, &c->thr, &c->pathPDF, &c->prevPDF, &c->wvlPDF, &c->lastPos, &c->shO, &c->shD, &c->shXYZ, &c->iterXYZ, &c->prevAcc,
						   &c->vxP, &c->vxN, &c->vxNx, &c->vxNy, &c->vxD };
	for (auto* b : f4)
		CU(b->alloc(n));
	CU(c->hit.alloc(n));
	CU(c->hitT.alloc(n));
	if (c->S.nLPE) {
		CU(c->lpeState.alloc(n));
		CU(c->lpeAcc.alloc(n * c->S.nLPE));
		CU(c->lpePrev.alloc(n * c->S.nLPE));
	}
	CU(cudaStreamSynchronize(c->stream));
	c->cachedTiles.assign(tiles, tiles + n_tiles);
	c->nSlots = (uint32_t)n;
	c->stateVersion++;
	if (c->stagedAuto) { // another wave size: measure again
		c->tuneStep = 0;
		c->tuneMs[0] = c->tuneMs[1] = 0;
	}
	return PRB_OK;
}

// k_shade sorts a window of rounds * block slots by material per thread block; larger windows give more uniform warps but
// fewer blocks, so rounds is chosen such that the grid still holds >= PRB_SHADE_FILL blocks per SM (measured on complex.prc,
// 2 M slots: windows of 8 x 512 slots with 2 blocks per SM shade 10 % faster than 4 x 512 with 4)
static void launchShadeOnly(prb_ctx* c, const WFState& W, cudaStream_t s);
// shade + regenerate: k_regen starts the next camera sample of every path that k_shade ended (dense list, see k_shade)
static void launchShade(prb_ctx* c, const WFState& W, cudaStream_t s)
{
	launchShadeOnly(c, W, s);
	if (!W.regenInTrace) // small scenes: k_trace_small regenerates the flagged slots in its prologue
		k_regen<<<(int)((c->nSlots + 127) / 128), 128, 0, s>>>(c->S, W);
}
// staged shading: k_shade_geom, then one k_shade_nee / k_shade_scatter launch per material TYPE present in the scene over that
// type's queue (grids sized for the worst case; blocks past the end of a queue return at once)
static void launchShadeStaged(prb_ctx* c, const WFState& W, cudaStream_t s)
{
	if (c->S.nLPE)
		k_shade_geom<true><<<(int)((c->nSlots + 127) / 128), 128, 0, s>>>(c->S, W);
	else
		k_shade_geom<false><<<(int)((c->nSlots + 127) / 128), 128, 0, s>>>(c->S, W);
	for (uint32_t t = 0; t < (uint32_t)SHADE_QUEUES; ++t) {
		const uint32_t q = W.queueOfType[t];
		if (q == 0xFF)
			continue;
		switch (t) {
		case PRB_MAT_DIFFUSE:
			if (c->hasImageNodes)
				launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_DIFFUSE>(c, W, q, s);
			else
				launchStageKernels<SHADE_MATERIALS_LAMBERT>(c, W, q, s);
			break;
		case PRB_MAT_DIELECTRIC: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_DIELECTRIC>(c, W, q, s); break;
		case PRB_MAT_CONDUCTOR: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_CONDUCTOR>(c, W, q, s); break;
		case PRB_MAT_ROUGHCONDUCTOR: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_ROUGHCONDUCTOR>(c, W, q, s); break;
		case PRB_MAT_ROUGHDIELECTRIC: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_ROUGHDIELECTRIC>(c, W, q, s); break;
		case PRB_MAT_PRINCIPLED: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_PRINCIPLED>(c, W, q, s); break;
		case PRB_MAT_MIRROR: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_MIRROR>(c, W, q, s); break;
		case PRB_MAT_ORENNAYAR: launchStageKernels<SHADE_MATERIALS_TYPE + PRB_MAT_ORENNAYAR>(c, W, q, s); break;
		default: launchStageKernels<SHADE_MATERIALS_COMBINED>(c, W, q, s); break; // blend / add: children of any leaf type
		}
	}
}
static void launchShadeOnly(prb_ctx* c, const WFState& W, cudaStream_t s)
{
	if (c->staged) {
		launchShadeStaged(c, W, s);
		return;
	}
	const bool combined = c->S.hasCombined != 0; // a scene with blend / add materials always mixes material types
	if (!c->mixedMaterials && !combined) {
		const int grid = (int)((c->nSlots + SHADE_BLOCK_UNIFORM - 1) / SHADE_BLOCK_UNIFORM);
		if (c->allLambert)
			k_shade<SHADE_BLOCK_UNIFORM, 1, SHADE_MATERIALS_LAMBERT><<<grid, SHADE_BLOCK_UNIFORM, 0, s>>>(c->S, W, 1);
		else
			k_shade<SHADE_BLOCK_UNIFORM, 1, SHADE_MATERIALS_LEAF><<<grid, SHADE_BLOCK_UNIFORM, 0, s>>>(c->S, W, 1);
		return;
	}
#ifndef PRB_SHADE_FILL
#define PRB_SHADE_FILL 2 /* blocks per SM the grid must still hold when a window spans several passes */
#endif
	const size_t perRound = (size_t)512 * c->smCount * PRB_SHADE_FILL;
	const int rounds	  = (int)std::max<size_t>(1, std::min<size_t>(SHADE_ROUNDS_MIXED, c->nSlots / perRound));
	const size_t window	  = (size_t)rounds * SHADE_BLOCK_MIXED;
	const int grid		  = (int)((c->nSlots + window - 1) / window);
	if (combined)
		k_shade<SHADE_BLOCK_MIXED, SHADE_ROUNDS_MIXED, SHADE_MATERIALS_COMBINED><<<grid, SHADE_BLOCK_MIXED, 0, s>>>(c->S, W, rounds);
	else
		k_shade<SHADE_BLOCK_MIXED, SHADE_ROUNDS_MIXED, SHADE_MATERIALS_LEAF><<<grid, SHADE_BLOCK_MIXED, 0, s>>>(c->S, W, rounds);
}
// one wavefront iteration; `iteration` alternates the counter of the compacted small-scene mode (WFState::parity)
static void launchShade(prb_ctx* c, const WFState& W, cudaStream_t s);
static void launchTrace(prb_ctx* c, const WFState& W, int blocks, cudaStream_t s);
static void launchIteration(prb_ctx* c, WFState W, int blocks, cudaStream_t s, int iteration, bool shade = true)
{
	W.parity = (uint32_t)(iteration & 1);
	launchTrace(c, W, blocks, s);
	if (shade)
		launchShade(c, W, s);
}
static void launchTrace(prb_ctx* c, const WFState& W, int blocks, cudaStream_t s)
{
	if (c->persistentTrace) {
		k_compact_active<<<(int)((c->nSlots + 1023) / 1024), 1024, 0, s>>>(W);
		k_trace<<<c->gridTrace, 128, 0, s>>>(c->S, W);
	} else if (c->smallScene)
		k_trace_small<<<(int)((c->nSlots + TRACE_SMALL_BLOCK - 1) / TRACE_SMALL_BLOCK), TRACE_SMALL_BLOCK, 0, s>>>(c->S, W);
	else
		k_trace_static<<<blocks, 128, 0, s>>>(c->S, W);
}

static WFState makeWF(prb_ctx* c, uint32_t first, uint32_t count)
{
	WFState W{};
	W.pixel		  = c->pixel.p;
	W.iter		  = c->iter.p;
	W.rayO		  = c->rayO.p;
	W.rayD		  = c->rayD.p;
	W.wvl		  = c->wvl.p;
	W.flagsDepth  = c->flagsDepth.p;
	W.thr		  = c->thr.p;
	W.pathPDF	  = c->pathPDF.p;
	W.prevPDF	  = c->prevPDF.p;
	W.wvlPDF	  = c->wvlPDF.p;
	W.lastPos	  = c->lastPos.p;
	W.hit		  = c->hit.p;
	W.hitT		  = c->hitT.p;
	W.shO		  = c->shO.p;
	W.shD		  = c->shD.p;
	W.shXYZ		  = c->shXYZ.p;
	W.iterXYZ	  = c->iterXYZ.p;
	W.prevAcc	  = c->prevAcc.p;
	W.state		  = c->slotState.p;
	W.counters	  = c->counters.p;
	W.regenList	  = c->regenList.p;
	W.activeList  = c->activeList.p;
	W.neeList	  = c->neeList.p;
	W.scatterList = c->scatterList.p;
	W.vxP		  = c->vxP.p;
	W.vxN		  = c->vxN.p;
	W.vxNx		  = c->vxNx.p;
	W.vxNy		  = c->vxNy.p;
	W.vxD		  = c->vxD.p;
	std::memcpy(W.queueOfType, c->queueOfType, sizeof(W.queueOfType));
	W.lpeState		= c->lpeState.p;
	W.lpeAcc		= c->lpeAcc.p;
	W.lpePrev		= c->lpePrev.p;
	W.lpeFilm		= c->lpeFilm.p;
	W.lpeFilmStride = (size_t)c->S.settings.film_width * c->S.settings.film_height * 3;
	W.rng		  = c->rng.p;
	W.filmMean	  = c->filmMean.p;
	W.sampleCount = c->sampleCount.p;
	W.aov		  = c->wantAOV ? c->aov.p : nullptr;
	W.aovExt	  = c->aovExt.p;
	W.feedback	  = c->feedback.p;
	W.varMean	  = c->S.settings.want_variance ? c->varMean.p : nullptr;
	W.varVar	  = c->S.settings.want_variance ? c->varVar.p : nullptr;
	W.stats		  = c->stats.p;
	W.nSlots	  = c->nSlots;
	W.firstIter	  = first;
	W.endIter	  = first + count;
	W.regenInTrace = c->regenInTrace() ? 1u : 0u;
	W.useActiveList = c->persistentTrace ? 1u : 0u;
	W.compactSmall	= c->compactSmall() ? 1u : 0u;
	W.parity		= 0;
	return W;
}

// The integrators whose samples end at the first hit ('ao', 'vf'): exactly iteration_count iterations of one sample per slot,
// ITERS_PER_GRAPH to a CUDA graph; the kernels of the iterations past the end of the range find every slot done (CNT_END_ITER)
// and return at once.  begin() enqueues the per-render start after the counters are cleared; launch(parity, k) enqueues kernel k
// of an iteration, which counts as stage[k] under profiling; key names everything the captured launches depend on.
extern "C++" {
template <class Begin, class Launch>
static prb_status renderFirstHit(prb_ctx* c, uint32_t first, uint32_t count, int kernels, const int* stage, const uint64_t (&key)[7],
								 const Begin& begin, const Launch& launch)
{
	constexpr int ITERS_PER_GRAPH = 8;
	cudaStream_t s	 = c->stream;
	c->lastFirstIter = first;
	c->lastEndIter	 = first + count;
	CU(cudaEventRecord(c->evA, s));
	CU(cudaMemsetAsync(c->counters.p, 0, CNT__COUNT * sizeof(uint32_t), s));
	begin();
	CU(cudaGetLastError());
	const uint32_t rounds = (count + ITERS_PER_GRAPH - 1) / ITERS_PER_GRAPH;
	if (c->profiling) { // the same launches without graph replay, each bracketed by an event pair
		const prb_status ps = reserveProfEvents(c, 2 * (size_t)kernels);
		if (ps != PRB_OK)
			return ps;
		for (uint32_t r = 0; r < rounds * ITERS_PER_GRAPH; ++r)
			for (int k = 0; k < kernels; ++k) {
				CU(cudaEventRecord(c->profEvents[2 * k], s));
				launch(r & 1u, k);
				CU(cudaEventRecord(c->profEvents[2 * k + 1], s));
				CU(cudaGetLastError());
				CU(cudaEventSynchronize(c->profEvents[2 * k + 1]));
				float ms = 0;
				CU(cudaEventElapsedTime(&ms, c->profEvents[2 * k], c->profEvents[2 * k + 1]));
				c->stageMs[stage[k]] += ms;
				c->stageLaunches[stage[k]] += 1;
			}
	} else {
		// the kernels read the iteration range from device memory, so one graph serves every call until the key changes
		const prb_status gs = c->firstHitGraph.update(s, key, [&] {
			for (int r = 0; r < ITERS_PER_GRAPH; ++r)
				for (int k = 0; k < kernels; ++k)
					launch((uint32_t)(r & 1), k);
		});
		if (gs != PRB_OK)
			return gs;
		for (uint32_t r = 0; r < rounds; ++r)
			CU(cudaGraphLaunch(c->firstHitGraph.exec, s));
	}
	c->kernelLaunches += 1 + (uint64_t)kernels * ITERS_PER_GRAPH * rounds;
	c->wavefrontIterations += (uint64_t)ITERS_PER_GRAPH * rounds;
	CU(cudaEventRecord(c->evB, s));
	CU(cudaEventSynchronize(c->evB));
	CU(cudaEventElapsedTime(&c->lastMs, c->evA, c->evB));
	return PRB_OK;
}
}

// 'ao': k_ao_primary, k_ao_occlusion, k_ao_fold per iteration
static prb_status renderAO(prb_ctx* c, uint32_t first, uint32_t count)
{
	const uint32_t n = c->integrator.sample_count;
	if ((uint64_t)c->nSlots * n > 0xFFFFFFFFull)
		return fail(PRB_ERR_UNSUPPORTED, "'ao': owned pixels x sample_count exceeds the 32-bit work counter");
	CU(c->aoRng.alloc(c->nSlots));
	CU(c->aoOccluded.alloc(c->nSlots));
	CU(c->aoHits.alloc(c->nSlots));
	cudaStream_t s	 = c->stream;
	const WFState W	 = makeWF(c, first, count);
	AOState A{ c->aoRng.p, c->aoOccluded.p, c->aoHits.p, c->aoJump.p, n, 0 };
	const int blocks = (int)((c->nSlots + 127) / 128);
	auto launch		 = [&](uint32_t parity, int kernel) { // kernel 0: primary, 1: occlusion, 2: fold
		A.parity = parity;
		if (kernel == 0) {
			if (c->smallScene)
				k_ao_primary<true><<<blocks, 128, 0, s>>>(c->S, W, A);
			else
				k_ao_primary<false><<<blocks, 128, 0, s>>>(c->S, W, A);
		} else if (kernel == 1) {
			if (c->smallScene)
				k_ao_occlusion<true><<<c->gridAOSmall, 128, 0, s>>>(c->S, W, A);
			else
				k_ao_occlusion<false><<<c->gridAO, 128, 0, s>>>(c->S, W, A);
		} else {
			k_ao_fold<<<blocks, 128, 0, s>>>(c->S, W, A);
		}
	};
	static const int stage[3] = { PRB_STAGE_TRACE, PRB_STAGE_TRACE, PRB_STAGE_SHADE };
	const uint64_t key[7]	  = { PRB_INTEGRATOR_AO, c->stateVersion, (uint64_t)(c->smallScene ? 1u : 0u) | (c->wantAOV ? 2u : 0u), n,
								  (uint64_t)(uintptr_t)A.jump, (uint64_t)(uintptr_t)A.rng, (uint64_t)(uintptr_t)A.hits };
	return renderFirstHit(c, first, count, 3, stage, key, [&] { k_ao_begin<<<blocks, 128, 0, s>>>(W, A); }, launch);
}

// 'vf': k_vf per iteration
static prb_status renderVF(prb_ctx* c, uint32_t first, uint32_t count)
{
	cudaStream_t s		= c->stream;
	const WFState W		= makeWF(c, first, count);
	const uint32_t mode = c->integrator.mode;
	const int blocks	= (int)((c->nSlots + 127) / 128);
	auto launch			= [&](uint32_t, int) {
		if (c->smallScene)
			k_vf<true><<<blocks, 128, 0, s>>>(c->S, W, mode);
		else
			k_vf<false><<<blocks, 128, 0, s>>>(c->S, W, mode);
	};
	static const int stage[1] = { PRB_STAGE_TRACE };
	const uint64_t key[7] = { PRB_INTEGRATOR_VF, c->stateVersion, (uint64_t)(c->smallScene ? 1u : 0u) | (c->wantAOV ? 2u : 0u), mode, 0, 0, 0 };
	return renderFirstHit(c, first, count, 1, stage, key, [&] { k_vf_begin<<<blocks, 128, 0, s>>>(W); }, launch);
}

prb_status prb_set_integrator(prb_ctx* c, const prb_integrator* in)
{
	if (!c || !in)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (in->type != PRB_INTEGRATOR_DIRECT && in->type != PRB_INTEGRATOR_AO && in->type != PRB_INTEGRATOR_VF)
		return fail(PRB_ERR_INVALID_ARG, "unknown integrator type " + std::to_string(in->type));
	if (in->type == PRB_INTEGRATOR_VF) {
		if (in->mode >= PRB_VF__COUNT)
			return fail(PRB_ERR_INVALID_ARG, "unknown 'vf' mode " + std::to_string(in->mode));
		if (c->S.nLPE)
			return fail(PRB_ERR_UNSUPPORTED, "'vf' does not fill light path expression channels");
	}
	if (in->type == PRB_INTEGRATOR_AO) {
		if (in->sample_count == 0)
			return fail(PRB_ERR_INVALID_ARG, "'ao' needs sample_count >= 1");
		if (c->S.nLPE)
			return fail(PRB_ERR_UNSUPPORTED, "'ao' does not fill light path expression channels");
		// jump[j] = M^(2j) mod 2^64: the pcg32_fast state after the two draws of each of j occlusion rays is s * jump[j]
		std::vector<uint64_t> jump(in->sample_count + 1);
		uint64_t m = 1;
		for (auto& v : jump) {
			v = m;
			m *= 6364136223846793005ULL * 6364136223846793005ULL;
		}
		CU(cudaSetDevice(c->device));
		CU(c->aoJump.upload(jump.data(), jump.size(), c->stream));
		CU(cudaStreamSynchronize(c->stream));
	}
	c->integrator = *in;
	return PRB_OK;
}
prb_status prb_get_integrator(prb_ctx* c, prb_integrator* out)
{
	if (!c || !out)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	*out = c->integrator;
	return PRB_OK;
}

prb_status prb_render_tiles(prb_ctx* c, const prb_tile* tiles, size_t n_tiles, uint32_t first_iteration, uint32_t iteration_count)
{
	if (!c || !tiles)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n_tiles == 0 || iteration_count == 0)
		return PRB_OK;
	if (!c->rngUploaded)
		return fail(PRB_ERR_INVALID_ARG, "prb_upload_rng has not been called for this scene (all-zero pcg32_fast states never advance)");
	CU(cudaSetDevice(c->device));
	prb_status st = setupSlots(c, tiles, n_tiles);
	if (st != PRB_OK)
		return st;
	if (c->integrator.type == PRB_INTEGRATOR_AO)
		return renderAO(c, first_iteration, iteration_count);
	if (c->integrator.type == PRB_INTEGRATOR_VF)
		return renderVF(c, first_iteration, iteration_count);
	cudaStream_t s = c->stream;
	const WFState W	 = makeWF(c, first_iteration, iteration_count);
	const int blocks = (int)((c->nSlots + 127) / 128);
	c->lastFirstIter = first_iteration;
	c->lastEndIter	 = first_iteration + iteration_count;
	CU(cudaEventRecord(c->evA, s));
	CU(cudaMemsetAsync(c->counters.p, 0, CNT__COUNT * sizeof(uint32_t), s));
	k_init_slots<<<blocks, 128, 0, s>>>(c->S, W);
	c->kernelLaunches += 1;
	CU(cudaGetLastError());
	// one wavefront iteration = k_trace + k_shade.  ITERS_PER_GRAPH iterations form one CUDA graph that is replayed;
	// the retired-slot counter is read back every GRAPHS_PER_POLL replays.
	constexpr int ITERS_PER_GRAPH = 8, GRAPHS_PER_POLL = 4;
	// upper bound on wavefront iterations: every sample needs at most max_ray_depth + 1 iterations
	const uint64_t maxIters = (uint64_t)iteration_count * (c->S.settings.max_ray_depth + 2) + 8;
	uint64_t done = 0;
	bool finished = false;
	auto poll = [&]() -> cudaError_t {
		cudaError_t e = cudaMemcpyAsync(c->hostCounters, c->counters.p, CNT__COUNT * sizeof(uint32_t), cudaMemcpyDeviceToHost, s);
		if (e == cudaSuccess)
			e = cudaStreamSynchronize(s);
		finished = c->hostCounters[CNT_RETIRED] >= c->nSlots;
		return e;
	};
	if (c->profiling) {
		// same launch sequence without graph replay, every kernel bracketed by an event pair on the context stream
		const prb_status ps = reserveProfEvents(c, (size_t)ITERS_PER_GRAPH * GRAPHS_PER_POLL * PRB_STAGE__COUNT * 2);
		if (ps != PRB_OK)
			return ps;
		while (!finished && done < maxIters + ITERS_PER_GRAPH * GRAPHS_PER_POLL) {
			size_t ne = 0;
			for (int r = 0; r < ITERS_PER_GRAPH * GRAPHS_PER_POLL; ++r) {
				WFState Wi = W;
				Wi.parity  = (uint32_t)(r & 1);
				CU(cudaEventRecord(c->profEvents[ne++], s));
				launchTrace(c, Wi, blocks, s);
				CU(cudaEventRecord(c->profEvents[ne++], s));
				CU(cudaEventRecord(c->profEvents[ne++], s));
				launchShade(c, Wi, s);
				CU(cudaEventRecord(c->profEvents[ne++], s));
				CU(cudaGetLastError());
			}
			done += ITERS_PER_GRAPH * GRAPHS_PER_POLL;
			c->kernelLaunches += c->launchesPerIteration(c->staged) * ITERS_PER_GRAPH * GRAPHS_PER_POLL;
			CU(poll());
			for (size_t i = 0; i + 1 < ne; i += 2) {
				float ms = 0;
				CU(cudaEventElapsedTime(&ms, c->profEvents[i], c->profEvents[i + 1]));
				const int stage = (int)((i / 2) % PRB_STAGE__COUNT);
				c->stageMs[stage] += ms;
				c->stageLaunches[stage] += 1;
			}
		}
	} else {
		// Undecided contexts time poll intervals in the order single, staged, staged, single (the number of live paths falls
		// slowly over a render; the symmetric order cancels that drift) and keep the faster path from then on.  Both leave the
		// same wavefront state behind every iteration, so they can alternate freely.
		static const bool tuneOrder[4] = { false, true, true, false };
		while (!finished && done < maxIters + ITERS_PER_GRAPH * GRAPHS_PER_POLL) {
			const bool tuning = c->stagedAuto && c->tuneStep < 4;
			const bool mode	  = tuning ? tuneOrder[c->tuneStep] : c->staged;
			// the kernels of the graph read the iteration range from device memory (CNT_END_ITER, written by k_init_slots), so one
			// instantiated graph serves every call until the scene, the slot buffers or the kernel variant change
			const uint64_t key[7] = { (c->stateVersion << 4) | (c->persistentTrace ? 1u : 0u) | (c->wantAOV ? 2u : 0u) | (c->smallScene ? 4u : 0u) | (mode ? 8u : 0u) };
			CachedGraph& graph	  = c->directGraph[mode ? 1 : 0];
			const prb_status gs	  = graph.update(s, key, [&] {
				const bool keep = c->staged; // the launches read the shading mode from the context
				c->staged		= mode;
				for (int r = 0; r < ITERS_PER_GRAPH; ++r)
					launchIteration(c, W, blocks, s, r);
				c->staged = keep;
			});
			if (gs != PRB_OK)
				return gs;
			cudaError_t e = cudaSuccess;
			if (tuning)
				e = cudaEventRecord(c->evT0, s);
			for (int r = 0; r < GRAPHS_PER_POLL && e == cudaSuccess; ++r)
				e = cudaGraphLaunch(graph.exec, s);
			if (tuning && e == cudaSuccess)
				e = cudaEventRecord(c->evT1, s);
			done += ITERS_PER_GRAPH * GRAPHS_PER_POLL;
			c->kernelLaunches += c->launchesPerIteration(mode) * ITERS_PER_GRAPH * GRAPHS_PER_POLL;
			if (e == cudaSuccess)
				e = poll();
			if (e != cudaSuccess)
				return fail(PRB_ERR_CUDA, std::string("wavefront loop failed: ") + cudaGetErrorString(e));
			if (tuning) {
				float ms = 0;
				CU(cudaEventElapsedTime(&ms, c->evT0, c->evT1));
				c->tuneMs[mode ? 1 : 0] += ms;
				if (++c->tuneStep == 4) {
					c->staged	  = c->tuneMs[1] < c->tuneMs[0];
					c->stagedAuto = false;
				}
			}
		}
	}
	// flush: samples that ended with their last shadow ray in flight are folded into the film by k_trace
	launchIteration(c, W, blocks, s, 0, false); // (an even number of iterations has run: parity 0)
	c->kernelLaunches += 1;
	CU(cudaGetLastError());
	c->wavefrontIterations += done;
	CU(cudaEventRecord(c->evB, s));
	CU(cudaEventSynchronize(c->evB));
	CU(cudaEventElapsedTime(&c->lastMs, c->evA, c->evB));
	if (!finished)
		return fail(PRB_ERR_CUDA, "wavefront loop did not terminate within the iteration bound");
	return PRB_OK;
}

prb_status prb_sync(prb_ctx* c)
{
	if (!c)
		return fail(PRB_ERR_INVALID_ARG, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}

static prb_status filteredFilm(prb_ctx* c, float** out, float* film = nullptr)
{
	if (!film)
		film = c->filmMean.p;
	const prb_settings& st = c->S.settings;
	const int r			   = st.filter_radius;
	bool identity		   = true; // centre weight 1, everything else <= eps (e.g. mitchell radius 1)
	if (r > 0)
		identity = false;
	if (identity) {
		*out = film;
		return PRB_OK;
	}
	k_filter<<<c->smCount * 4, 256, 0, c->stream>>>(film, c->filmTmp.p, (int)st.film_width, (int)st.film_height, r, c->pool.p + st.filter_offset);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	*out = c->filmTmp.p;
	return PRB_OK;
}

prb_status prb_film_download(prb_ctx* c, float* xyz, uint32_t* sample_count)
{
	if (!c || !c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	if (xyz) {
		float* src = nullptr;
		prb_status st = filteredFilm(c, &src);
		if (st != PRB_OK)
			return st;
		CU(cudaMemcpyAsync(xyz, src, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	}
	if (sample_count)
		CU(cudaMemcpyAsync(sample_count, c->sampleCount.p, npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_download_aov(prb_ctx* c, float* aov10)
{
	if (!c || !c->haveScene || !aov10)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	CU(cudaMemcpyAsync(aov10, c->aov.p, npix * 10 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_download_feedback(prb_ctx* c, uint32_t* feedback)
{
	if (!c || !c->haveScene || !feedback)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	CU(cudaMemcpyAsync(feedback, c->feedback.p, npix * sizeof(uint32_t), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_download_variance(prb_ctx* c, float* online_mean, float* online_variance)
{
	if (!c || !c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (!c->S.settings.want_variance || !c->varMean.p)
		return fail(PRB_ERR_UNSUPPORTED, "the scene was uploaded without prb_settings.want_variance");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	if (online_mean)
		CU(cudaMemcpyAsync(online_mean, c->varMean.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	if (online_variance)
		CU(cudaMemcpyAsync(online_variance, c->varVar.p, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_download_aov_ext(prb_ctx* c, float* aov11)
{
	if (!c || !c->haveScene || !aov11)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	if (!c->aovExt.p)
		return fail(PRB_ERR_UNSUPPORTED, "the scene was uploaded without prb_settings.want_aov_ext");
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	CU(cudaMemcpyAsync(aov11, c->aovExt.p, npix * PRB_AOV_EXT * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_download_lpe(prb_ctx* c, uint32_t index, float* xyz)
{
	if (!c || !c->haveScene || !xyz)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	if (index >= c->S.nLPE || !c->lpeFilm.p)
		return fail(PRB_ERR_INVALID_ARG, "the scene has no light path expression " + std::to_string(index));
	CU(cudaSetDevice(c->device));
	const size_t npix = (size_t)c->S.settings.film_width * c->S.settings.film_height;
	float* src		  = nullptr;
	prb_status st	  = filteredFilm(c, &src, c->lpeFilm.p + (size_t)index * npix * 3);
	if (st != PRB_OK)
		return st;
	CU(cudaMemcpyAsync(xyz, src, npix * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_export_device(prb_ctx* c, float* device_dst)
{
	if (!c || !c->haveScene || !device_dst)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	CU(cudaSetDevice(c->device));
	const uint32_t npix = c->S.settings.film_width * c->S.settings.film_height;
	k_film_export<<<c->smCount * 4, 256, 0, c->stream>>>(c->filmMean.p, c->sampleCount.p, device_dst, npix);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_film_import_device(prb_ctx* c, const float* device_src)
{
	if (!c || !c->haveScene || !device_src)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded / null buffer");
	CU(cudaSetDevice(c->device));
	const uint32_t npix = c->S.settings.film_width * c->S.settings.film_height;
	k_film_import<<<c->smCount * 4, 256, 0, c->stream>>>(device_src, c->filmMean.p, c->sampleCount.p, npix);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}

// ------------------------------------------------------------------ multi-GPU film combine
namespace {
// the handful of NCCL entry points used, resolved at run time from libnccl.so.2 (no link-time dependency: a single-GPU
// client never needs the library)
struct NcclUniqueId {
	char internal[128];
};
struct NcclApi {
	void* lib = nullptr;
	int (*GetUniqueId)(NcclUniqueId*)														   = nullptr;
	int (*CommInitRank)(void**, int, NcclUniqueId, int)										   = nullptr;
	int (*CommDestroy)(void*)																   = nullptr;
	int (*Reduce)(const void*, void*, size_t, int /*dtype*/, int /*op*/, int, void*, cudaStream_t) = nullptr;
	int (*GroupStart)()																		   = nullptr;
	int (*GroupEnd)()																		   = nullptr;
	const char* (*GetErrorString)(int)														   = nullptr;
	bool ok() const { return GetUniqueId && CommInitRank && CommDestroy && Reduce && GroupStart && GroupEnd && GetErrorString; }
};
constexpr int NCCL_FLOAT32 = 7, NCCL_UINT32 = 3, NCCL_SUM = 0; // ncclDataType_t / ncclRedOp_t values (stable since NCCL 2.0)
NcclApi& nccl()
{
	static NcclApi api = [] {
		NcclApi a;
		// RTLD_NOLOAD first: reuse the copy the process already holds (torch ships its own), else the system library
		a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);
		if (!a.lib)
			a.lib = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
		if (!a.lib)
			a.lib = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
		if (a.lib) {
			a.GetUniqueId	 = reinterpret_cast<decltype(a.GetUniqueId)>(dlsym(a.lib, "ncclGetUniqueId"));
			a.CommInitRank	 = reinterpret_cast<decltype(a.CommInitRank)>(dlsym(a.lib, "ncclCommInitRank"));
			a.CommDestroy	 = reinterpret_cast<decltype(a.CommDestroy)>(dlsym(a.lib, "ncclCommDestroy"));
			a.Reduce		 = reinterpret_cast<decltype(a.Reduce)>(dlsym(a.lib, "ncclReduce"));
			a.GroupStart	 = reinterpret_cast<decltype(a.GroupStart)>(dlsym(a.lib, "ncclGroupStart"));
			a.GroupEnd		 = reinterpret_cast<decltype(a.GroupEnd)>(dlsym(a.lib, "ncclGroupEnd"));
			a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(dlsym(a.lib, "ncclGetErrorString"));
		}
		return a;
	}();
	return api;
}
#define NC(x)                                                                                                 \
	do {                                                                                                      \
		int r_ = (x);                                                                                         \
		if (r_ != 0)                                                                                          \
			return fail(PRB_ERR_CUDA, std::string(#x) + ": " + nccl().GetErrorString(r_));                    \
	} while (0)

float partitionWeight(const prb_ctx* c, int partition, uint32_t totalIterations)
{ // PRB_PARTITION_SAMPLES: the context's film is sum / lastEndIter (it started from an empty film at lastFirstIter)
	if (partition != PRB_PARTITION_SAMPLES || totalIterations == 0)
		return 1.0f;
	return (float)c->lastEndIter / (float)totalIterations;
}
} // namespace

prb_status prb_comm_unique_id(uint8_t id[PRB_COMM_UNIQUE_ID_BYTES])
{
	if (!id)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!nccl().ok())
		return fail(PRB_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded");
	NcclUniqueId u;
	NC(nccl().GetUniqueId(&u));
	static_assert(sizeof(u) == PRB_COMM_UNIQUE_ID_BYTES, "ncclUniqueId is 128 bytes");
	std::memcpy(id, &u, sizeof(u));
	return PRB_OK;
}
prb_status prb_comm_init(prb_ctx* c, const uint8_t id[PRB_COMM_UNIQUE_ID_BYTES], int rank, int world)
{
	if (!c || !id || world < 1 || rank < 0 || rank >= world)
		return fail(PRB_ERR_INVALID_ARG, "invalid communicator arguments");
	if (!nccl().ok())
		return fail(PRB_ERR_UNSUPPORTED, "libnccl.so.2 could not be loaded");
	CU(cudaSetDevice(c->device));
	prb_comm_destroy(c);
	NcclUniqueId u;
	std::memcpy(&u, id, sizeof(u));
	NC(nccl().CommInitRank(&c->ncclComm, world, u, rank));
	c->commRank	 = rank;
	c->commWorld = world;
	return PRB_OK;
}
prb_status prb_comm_destroy(prb_ctx* c)
{
	if (!c)
		return fail(PRB_ERR_INVALID_ARG, "null context");
	if (c->ncclComm) {
		cudaSetDevice(c->device);
		cudaStreamSynchronize(c->stream);
		nccl().CommDestroy(c->ncclComm);
		c->ncclComm = nullptr;
	}
	c->commRank	 = 0;
	c->commWorld = 1;
	return PRB_OK;
}
prb_status prb_film_reduce_comm(prb_ctx* c, int partition, uint32_t total_iterations, int root)
{
	if (!c || !c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (partition != PRB_PARTITION_TILES && partition != PRB_PARTITION_SAMPLES)
		return fail(PRB_ERR_INVALID_ARG, "partition must be PRB_PARTITION_TILES or PRB_PARTITION_SAMPLES");
	if (!c->ncclComm)
		return fail(PRB_ERR_INVALID_ARG, "prb_comm_init has not been called");
	if (root < 0 || root >= c->commWorld)
		return fail(PRB_ERR_INVALID_ARG, "root out of range");
	CU(cudaSetDevice(c->device));
	const uint32_t npix = c->S.settings.film_width * c->S.settings.film_height;
	CU(c->reduceF.alloc((size_t)npix * FILM_PACK));
	CU(c->reduceU.alloc(npix));
	cudaStream_t s = c->stream;
	CU(cudaEventRecord(c->evA, s));
	k_film_pack<<<c->smCount * 4, 256, 0, s>>>(c->filmMean.p, c->sampleCount.p, c->aov.p, c->feedback.p, partitionWeight(c, partition, total_iterations), c->reduceF.p,
												c->reduceU.p, npix);
	CU(cudaGetLastError());
	if (c->lpeFilm.p) {
		const float w = partitionWeight(c, partition, total_iterations);
		if (w != 1.0f) {
			k_scale_add<<<c->smCount * 4, 256, 0, s>>>(c->lpeFilm.p, nullptr, w, 0.0f, (size_t)npix * 3 * c->S.nLPE);
			c->kernelLaunches += 1;
		}
	}
	NC(nccl().GroupStart());
	NC(nccl().Reduce(c->reduceF.p, c->reduceF.p, (size_t)npix * FILM_PACK, NCCL_FLOAT32, NCCL_SUM, root, c->ncclComm, s));
	NC(nccl().Reduce(c->reduceU.p, c->reduceU.p, npix, NCCL_UINT32, NCCL_SUM, root, c->ncclComm, s));
	if (c->varMean.p && partition == PRB_PARTITION_TILES) { // disjoint pixel ownership: the sum is the owner's value
		NC(nccl().Reduce(c->varMean.p, c->varMean.p, (size_t)npix * 3, NCCL_FLOAT32, NCCL_SUM, root, c->ncclComm, s));
		NC(nccl().Reduce(c->varVar.p, c->varVar.p, (size_t)npix * 3, NCCL_FLOAT32, NCCL_SUM, root, c->ncclComm, s));
	}
	// the extended AOV sums add up like the ten packed ones; the expression channels are films: weighted like the main one
	if (c->aovExt.p)
		NC(nccl().Reduce(c->aovExt.p, c->aovExt.p, (size_t)npix * PRB_AOV_EXT, NCCL_FLOAT32, NCCL_SUM, root, c->ncclComm, s));
	if (c->lpeFilm.p)
		NC(nccl().Reduce(c->lpeFilm.p, c->lpeFilm.p, (size_t)npix * 3 * c->S.nLPE, NCCL_FLOAT32, NCCL_SUM, root, c->ncclComm, s));
	NC(nccl().GroupEnd());
	c->kernelLaunches += 1;
	if (c->commRank == root) {
		k_film_unpack<<<c->smCount * 4, 256, 0, s>>>(c->reduceF.p, c->reduceU.p, c->filmMean.p, c->sampleCount.p, c->aov.p, c->feedback.p, npix);
		CU(cudaGetLastError());
		c->kernelLaunches += 1;
	}
	CU(cudaEventRecord(c->evB, s));
	CU(cudaEventSynchronize(c->evB));
	CU(cudaEventElapsedTime(&c->lastReduceMs, c->evA, c->evB));
	return PRB_OK;
}
prb_status prb_film_reduce(prb_ctx** ctxs, int n, int partition)
{
	if (!ctxs || n < 1 || n > PEER_MAX + 1)
		return fail(PRB_ERR_INVALID_ARG, "1 .. 16 contexts expected");
	if (partition != PRB_PARTITION_TILES && partition != PRB_PARTITION_SAMPLES)
		return fail(PRB_ERR_INVALID_ARG, "partition must be PRB_PARTITION_TILES or PRB_PARTITION_SAMPLES");
	prb_ctx* root = ctxs[0];
	uint32_t total = 0;
	for (int i = 0; i < n; ++i) {
		if (!ctxs[i] || !ctxs[i]->haveScene)
			return fail(PRB_ERR_NO_SCENE, "a context has no scene");
		if (ctxs[i]->S.settings.film_width != root->S.settings.film_width || ctxs[i]->S.settings.film_height != root->S.settings.film_height)
			return fail(PRB_ERR_INVALID_ARG, "contexts render films of different sizes");
		for (int j = 0; j < i; ++j)
			if (ctxs[j] == ctxs[i])
				return fail(PRB_ERR_INVALID_ARG, "a context is listed twice");
		total += ctxs[i]->lastEndIter - ctxs[i]->lastFirstIter;
	}
	if (n == 1)
		return PRB_OK;
	const uint32_t npix = root->S.settings.film_width * root->S.settings.film_height;
	PeerFilms P{};
	P.n			 = n - 1;
	P.rootWeight = partitionWeight(root, partition, total);
	// every contributing film must be complete before the root reads it
	for (int i = 1; i < n; ++i) {
		CU(cudaSetDevice(ctxs[i]->device));
		CU(cudaStreamSynchronize(ctxs[i]->stream));
	}
	CU(cudaSetDevice(root->device));
	std::vector<DBuf<float>> stageF(n);
	std::vector<DBuf<uint32_t>> stageU(n);
	for (int i = 1; i < n; ++i) {
		prb_ctx* p	 = ctxs[i];
		bool direct = p->device == root->device;
		if (!direct) {
			int can = 0;
			CU(cudaDeviceCanAccessPeer(&can, root->device, p->device));
			if (can) {
				const cudaError_t e = cudaDeviceEnablePeerAccess(p->device, 0);
				if (e == cudaSuccess || e == cudaErrorPeerAccessAlreadyEnabled) {
					cudaGetLastError();
					direct = true;
				}
			}
		}
		if (direct) { // the gather kernel loads the peer's film through NVLink
			P.mean[i - 1]	  = p->filmMean.p;
			P.count[i - 1]	  = p->sampleCount.p;
			P.aov[i - 1]	  = p->aov.p;
			P.feedback[i - 1] = p->feedback.p;
		} else { // no peer access: stage the film on the root device
			CU(stageF[i].alloc((size_t)npix * 13));
			CU(stageU[i].alloc((size_t)npix * 2));
			CU(cudaMemcpyPeerAsync(stageF[i].p, root->device, p->filmMean.p, p->device, (size_t)npix * 3 * sizeof(float), root->stream));
			CU(cudaMemcpyPeerAsync(stageF[i].p + (size_t)npix * 3, root->device, p->aov.p, p->device, (size_t)npix * 10 * sizeof(float), root->stream));
			CU(cudaMemcpyPeerAsync(stageU[i].p, root->device, p->sampleCount.p, p->device, (size_t)npix * sizeof(uint32_t), root->stream));
			CU(cudaMemcpyPeerAsync(stageU[i].p + npix, root->device, p->feedback.p, p->device, (size_t)npix * sizeof(uint32_t), root->stream));
			P.mean[i - 1]	  = stageF[i].p;
			P.aov[i - 1]	  = stageF[i].p + (size_t)npix * 3;
			P.count[i - 1]	  = stageU[i].p;
			P.feedback[i - 1] = stageU[i].p + npix;
		}
		P.weight[i - 1] = partitionWeight(p, partition, total);
	}
	CU(cudaEventRecord(root->evA, root->stream));
	k_film_gather<<<root->smCount * 4, 256, 0, root->stream>>>(P, root->filmMean.p, root->sampleCount.p, root->aov.p, root->feedback.p, npix);
	root->kernelLaunches += 1;
	CU(cudaGetLastError());
	{ // extended AOV sums and expression channels: one staged pass per peer and buffer
		const size_t nExt = root->aovExt.p ? (size_t)npix * PRB_AOV_EXT : 0, nLpe = root->lpeFilm.p ? (size_t)npix * 3 * root->S.nLPE : 0;
		DBuf<float> stage;
		CU(stage.alloc(std::max<size_t>(std::max(nExt, nLpe), 1)));
		if (nLpe && P.rootWeight != 1.0f) {
			k_scale_add<<<root->smCount * 4, 256, 0, root->stream>>>(root->lpeFilm.p, nullptr, P.rootWeight, 0.0f, nLpe);
			root->kernelLaunches += 1;
		}
		for (int i = 1; i < n; ++i) {
			if (nExt && ctxs[i]->aovExt.p) {
				CU(cudaMemcpyPeerAsync(stage.p, root->device, ctxs[i]->aovExt.p, ctxs[i]->device, nExt * sizeof(float), root->stream));
				k_add_buffer<<<root->smCount * 4, 256, 0, root->stream>>>(root->aovExt.p, stage.p, nExt);
				root->kernelLaunches += 1;
			}
			if (nLpe && ctxs[i]->lpeFilm.p && ctxs[i]->S.nLPE == root->S.nLPE) {
				CU(cudaMemcpyPeerAsync(stage.p, root->device, ctxs[i]->lpeFilm.p, ctxs[i]->device, nLpe * sizeof(float), root->stream));
				k_scale_add<<<root->smCount * 4, 256, 0, root->stream>>>(root->lpeFilm.p, stage.p, 1.0f, P.weight[i - 1], nLpe);
				root->kernelLaunches += 1;
			}
		}
		CU(cudaStreamSynchronize(root->stream));
	}
	if (root->varMean.p && partition == PRB_PARTITION_TILES) {
		DBuf<float> stage;
		CU(stage.alloc((size_t)npix * 3));
		for (int i = 1; i < n; ++i) {
			if (!ctxs[i]->varMean.p)
				continue;
			float* srcs[2] = { ctxs[i]->varMean.p, ctxs[i]->varVar.p };
			float* dsts[2] = { root->varMean.p, root->varVar.p };
			for (int k = 0; k < 2; ++k) {
				CU(cudaMemcpyPeerAsync(stage.p, root->device, srcs[k], ctxs[i]->device, (size_t)npix * 3 * sizeof(float), root->stream));
				k_add_buffer<<<root->smCount * 4, 256, 0, root->stream>>>(dsts[k], stage.p, (size_t)npix * 3);
				root->kernelLaunches += 1;
			}
		}
		CU(cudaStreamSynchronize(root->stream));
	}
	CU(cudaEventRecord(root->evB, root->stream));
	CU(cudaEventSynchronize(root->evB));
	CU(cudaEventElapsedTime(&root->lastReduceMs, root->evA, root->evB));
	return PRB_OK;
}
prb_status prb_last_reduce_ms(prb_ctx* c, float* ms)
{
	if (!c || !ms)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	*ms = c->lastReduceMs;
	return PRB_OK;
}

// ------------------------------------------------------------------ stream tracing
static prb_status traceDevice(prb_ctx* c, const prb_ray_soa* r, size_t n, prb_hit_soa* hits, uint8_t* occluded)
{
	CU(c->counters.alloc(CNT__COUNT));
	CU(cudaMemsetAsync(c->counters.p + CNT_WORK, 0, sizeof(uint32_t), c->stream));
	CU(cudaEventRecord(c->evA, c->stream));
	if (hits)
		k_trace_closest<<<c->gridTraceClosest, 128, 0, c->stream>>>(c->S, r->org_x, r->org_y, r->org_z, r->dir_x, r->dir_y, r->dir_z, r->tmin, r->tmax, (uint32_t)n,
																	 c->counters.p + CNT_WORK, hits->entity_id, hits->primitive_id, hits->u, hits->v, hits->t);
	else
		k_trace_any<<<c->gridTraceAny, 128, 0, c->stream>>>(c->S, r->org_x, r->org_y, r->org_z, r->dir_x, r->dir_y, r->dir_z, r->tmin, r->tmax, (uint32_t)n,
															 c->counters.p + CNT_WORK, occluded);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	CU(cudaEventRecord(c->evB, c->stream));
	CU(cudaEventSynchronize(c->evB));
	CU(cudaEventElapsedTime(&c->lastMs, c->evA, c->evB));
	return PRB_OK;
}
prb_status prb_trace_closest_device(prb_ctx* c, const prb_ray_soa* rays, size_t n, prb_hit_soa* hits)
{
	if (!c || !rays || !hits)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n == 0)
		return PRB_OK;
	CU(cudaSetDevice(c->device));
	return traceDevice(c, rays, n, hits, nullptr);
}
prb_status prb_trace_any_device(prb_ctx* c, const prb_ray_soa* rays, size_t n, uint8_t* occluded)
{
	if (!c || !rays || !occluded)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n == 0)
		return PRB_OK;
	CU(cudaSetDevice(c->device));
	return traceDevice(c, rays, n, nullptr, occluded);
}
static prb_status stageRays(prb_ctx* c, const prb_ray_soa* rays, size_t n, prb_ray_soa& dev)
{
	CU(c->scratchF.alloc(n * 8));
	const float* src[8] = { rays->org_x, rays->org_y, rays->org_z, rays->dir_x, rays->dir_y, rays->dir_z, rays->tmin, rays->tmax };
	const float* dst[8];
	for (int k = 0; k < 8; ++k) {
		if (!src[k]) {
			if (k < 6)
				return fail(PRB_ERR_INVALID_ARG, "ray origin/direction arrays must not be NULL");
			dst[k] = nullptr;
			continue;
		}
		CU(cudaMemcpyAsync(c->scratchF.p + k * n, src[k], n * sizeof(float), cudaMemcpyHostToDevice, c->stream));
		dst[k] = c->scratchF.p + k * n;
	}
	dev = prb_ray_soa{ dst[0], dst[1], dst[2], dst[3], dst[4], dst[5], dst[6], dst[7] };
	return PRB_OK;
}
prb_status prb_trace_closest(prb_ctx* c, const prb_ray_soa* rays, size_t n, prb_hit_soa* hits)
{
	if (!c || !rays || !hits)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n == 0)
		return PRB_OK;
	CU(cudaSetDevice(c->device));
	prb_ray_soa dr;
	prb_status st = stageRays(c, rays, n, dr);
	if (st != PRB_OK)
		return st;
	CU(c->scratchU.alloc(n * 5));
	prb_hit_soa dh{ c->scratchU.p, c->scratchU.p + n, reinterpret_cast<float*>(c->scratchU.p + 2 * n), reinterpret_cast<float*>(c->scratchU.p + 3 * n),
					reinterpret_cast<float*>(c->scratchU.p + 4 * n) };
	st = traceDevice(c, &dr, n, &dh, nullptr);
	if (st != PRB_OK)
		return st;
	CU(cudaMemcpyAsync(hits->entity_id, dh.entity_id, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(hits->primitive_id, dh.primitive_id, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(hits->u, dh.u, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(hits->v, dh.v, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(hits->t, dh.t, n * 4, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_trace_any(prb_ctx* c, const prb_ray_soa* rays, size_t n, uint8_t* occluded)
{
	if (!c || !rays || !occluded)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	if (n == 0)
		return PRB_OK;
	CU(cudaSetDevice(c->device));
	prb_ray_soa dr;
	prb_status st = stageRays(c, rays, n, dr);
	if (st != PRB_OK)
		return st;
	CU(c->scratchB.alloc(n));
	st = traceDevice(c, &dr, n, nullptr, c->scratchB.p);
	if (st != PRB_OK)
		return st;
	CU(cudaMemcpyAsync(occluded, c->scratchB.p, n, cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}

prb_status prb_generate_camera_rays(prb_ctx* c, const prb_tile* tiles, size_t n_tiles, uint32_t iteration, float* org_xyz, float* dir_xyz,
									float* wavelengths4, uint32_t* pixel_index, size_t capacity, size_t* n_out)
{
	if (!c || !tiles || !org_xyz || !dir_xyz || !wavelengths4 || !pixel_index || !n_out)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	CU(cudaSetDevice(c->device));
	const uint32_t W = c->S.settings.film_width, H = c->S.settings.film_height;
	std::vector<uint32_t> pix;
	for (size_t t = 0; t < n_tiles; ++t) {
		if (tiles[t].ex > W || tiles[t].ey > H)
			return fail(PRB_ERR_INVALID_ARG, "tile outside the film");
		for (uint32_t y = tiles[t].sy; y < tiles[t].ey; ++y)
			for (uint32_t x = tiles[t].sx; x < tiles[t].ex; ++x)
				if (pix.size() < capacity)
					pix.push_back(y * W + x);
	}
	const size_t n = pix.size();
	*n_out		   = n;
	if (n == 0)
		return PRB_OK;
	CU(c->scratchU.upload(pix.data(), n, c->stream));
	CU(c->scratchF.alloc(n * 10));
	float *dorg = c->scratchF.p, *ddir = c->scratchF.p + 3 * n, *dwvl = c->scratchF.p + 6 * n;
	k_camera_rays<<<c->smCount * 4, 256, 0, c->stream>>>(c->S, c->rng.p, c->scratchU.p, (uint32_t)n, iteration, dorg, ddir, dwvl);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	CU(cudaMemcpyAsync(org_xyz, dorg, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(dir_xyz, ddir, n * 3 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaMemcpyAsync(wavelengths4, dwvl, n * 4 * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	std::memcpy(pixel_index, pix.data(), n * sizeof(uint32_t));
	return PRB_OK;
}

static prb_status materialCall(prb_ctx* c, const prb_material_query* q, size_t n, prb_material_result* out, bool sample)
{
	if (!c || !q || !out)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	if (!c->haveScene)
		return fail(PRB_ERR_NO_SCENE, "no scene uploaded");
	for (size_t i = 0; i < n; ++i)
		if (q[i].material_id >= c->S.nMaterials)
			return fail(PRB_ERR_INVALID_ARG, "material id out of range");
	if (n == 0)
		return PRB_OK;
	CU(cudaSetDevice(c->device));
	CU(c->scratchQ.upload(q, n, c->stream));
	CU(c->scratchR.alloc(n));
	const int grid = (int)std::min<size_t>((n + 127) / 128, (size_t)c->smCount * 4);
	if (sample)
		k_material_sample<<<grid, 128, 0, c->stream>>>(c->S, c->scratchQ.p, (uint32_t)n, c->scratchR.p);
	else
		k_material_eval<<<grid, 128, 0, c->stream>>>(c->S, c->scratchQ.p, (uint32_t)n, c->scratchR.p);
	c->kernelLaunches++;
	CU(cudaGetLastError());
	CU(cudaMemcpyAsync(out, c->scratchR.p, n * sizeof(prb_material_result), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	return PRB_OK;
}
prb_status prb_material_eval(prb_ctx* c, const prb_material_query* q, size_t n, prb_material_result* out) { return materialCall(c, q, n, out, false); }
prb_status prb_material_sample(prb_ctx* c, const prb_material_query* q, size_t n, prb_material_result* out) { return materialCall(c, q, n, out, true); }

prb_status prb_get_stats(prb_ctx* c, prb_stats* out)
{
	if (!c || !out)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	CU(cudaSetDevice(c->device));
	unsigned long long h[ST__COUNT];
	CU(cudaMemcpyAsync(h, c->stats.p, sizeof(h), cudaMemcpyDeviceToHost, c->stream));
	CU(cudaStreamSynchronize(c->stream));
	out->camera_ray_count	  = h[ST_CAMERA_RAY];
	out->light_ray_count	  = h[ST_LIGHT_RAY];
	out->primary_ray_count	  = h[ST_PRIMARY];
	out->bounce_ray_count	  = h[ST_BOUNCE];
	out->shadow_ray_count	  = h[ST_SHADOW];
	out->monochrome_ray_count = h[ST_MONO];
	out->pixel_sample_count	  = h[ST_PIXEL_SAMPLE];
	out->entity_hit_count	  = h[ST_ENTITY_HIT];
	out->background_hit_count = h[ST_BG_HIT];
	out->camera_depth_count	  = h[ST_CAMERA_DEPTH];
	out->light_depth_count	  = h[ST_LIGHT_DEPTH];
	out->kernel_launches	  = c->kernelLaunches;
	out->wavefront_iterations = c->wavefrontIterations;
	return PRB_OK;
}
prb_status prb_reset_stats(prb_ctx* c)
{
	if (!c)
		return fail(PRB_ERR_INVALID_ARG, "null context");
	CU(cudaSetDevice(c->device));
	CU(cudaMemsetAsync(c->stats.p, 0, ST__COUNT * sizeof(unsigned long long), c->stream));
	c->kernelLaunches	   = 0;
	c->wavefrontIterations = 0;
	return PRB_OK;
}
prb_status prb_set_profiling(prb_ctx* c, int enabled)
{
	if (!c)
		return fail(PRB_ERR_INVALID_ARG, "null context");
	c->profiling = enabled != 0;
	for (int i = 0; i < PRB_STAGE__COUNT; ++i) {
		c->stageMs[i]		= 0;
		c->stageLaunches[i] = 0;
	}
	return PRB_OK;
}
prb_status prb_get_stage_times(prb_ctx* c, float* ms4, uint64_t* launches4)
{
	if (!c || !ms4 || !launches4)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	for (int i = 0; i < PRB_STAGE__COUNT; ++i) {
		ms4[i]		 = c->stageMs[i];
		launches4[i] = c->stageLaunches[i];
	}
	return PRB_OK;
}
prb_status prb_set_shading_mode(prb_ctx* c, int mode)
{
	if (!c || mode < PRB_SHADING_AUTO || mode > PRB_SHADING_STAGED)
		return fail(PRB_ERR_INVALID_ARG, "invalid shading mode");
	if (c->S.nLPE && mode != PRB_SHADING_STAGED)
		return fail(PRB_ERR_UNSUPPORTED, "scenes with light path expression channels shade staged");
	c->stagedAuto = mode == PRB_SHADING_AUTO && !c->allLambert;
	c->staged	  = mode == PRB_SHADING_STAGED;
	c->tuneStep	  = 0;
	c->tuneMs[0] = c->tuneMs[1] = 0;
	if (c->nSlots) { // the queues of the staged path are sized with the slots
		c->cachedTiles.clear();
		c->nSlots = 0;
	}
	return PRB_OK;
}
prb_status prb_get_shading_mode(prb_ctx* c, int* mode)
{
	if (!c || !mode)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	*mode = c->stagedAuto ? PRB_SHADING_AUTO : (c->staged ? PRB_SHADING_STAGED : PRB_SHADING_SINGLE);
	return PRB_OK;
}
prb_status prb_last_device_ms(prb_ctx* c, float* ms)
{
	if (!c || !ms)
		return fail(PRB_ERR_INVALID_ARG, "null argument");
	*ms = c->lastMs;
	return PRB_OK;
}
}
