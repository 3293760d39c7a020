// Flattens an Environment (scene database + settings) into the POD prb_scene_desc and builds the two-level
// BVH8 (TLAS over entities, one BLAS per mesh / plane).  This is the host half of what the reference does in
// Environment::createRenderFactory + Scene::setupScene + RenderContext::start (set-up only, no per-sample work).
#include "prh.h"

#include <chrono>

namespace PR {
void CompiledScene::finalize()
{
	desc.abi_version		= PRB_ABI_VERSION;
	desc.n_nodes			= (uint32)nodes.size();
	desc.nodes				= nodes.data();
	desc.n_materials		= (uint32)materials.size();
	desc.materials			= materials.data();
	desc.n_emissions		= (uint32)emissions.size();
	desc.emissions			= emissions.data();
	desc.n_entities			= (uint32)entities.size();
	desc.entities			= entities.data();
	desc.n_entity_materials = (uint32)entityMaterials.size();
	desc.entity_materials	= entityMaterials.data();
	desc.n_meshes			= (uint32)meshes.size();
	desc.meshes				= meshes.data();
	desc.n_vertices			= (uint32)(vertices.size() / 3);
	desc.vertices			= vertices.data();
	desc.normals			= normals.data();
	desc.uvs				= uvs.data();
	desc.n_faces			= (uint32)(faceIndices.size() / 4);
	desc.face_indices		= faceIndices.data();
	desc.face_slots			= faceSlots.data();
	desc.n_lights			= (uint32)lights.size();
	desc.lights				= lights.data();
	desc.light_cdf			= lightCDF.data();
	desc.n_bvh_nodes		= (uint32)bvhNodes.size();
	desc.bvh_nodes			= bvhNodes.data();
	desc.n_bvh_tris			= (uint32)bvhTris.size();
	desc.bvh_tris			= bvhTris.data();
	desc.n_tlas_refs		= (uint32)tlasRefs.size();
	desc.tlas_refs			= tlasRefs.data();
	desc.n_pool				= (uint32)pool.size();
	desc.pool				= pool.data();
	desc.n_lpe_bytes		= (uint32)lpeTables.size();
	desc.lpe_tables			= lpeTables.data();
}

static BoundingBox padBox(BoundingBox b)
{ // conservative padding against the ulp-level slack of the watertight triangle test
	float m = 0;
	for (int i = 0; i < 3; ++i)
		m = std::max(m, std::max(std::abs(b.lo[i]), std::abs(b.hi[i])));
	const float pad = std::max(1e-6f * m, 1e-30f);
	b.lo			= b.lo - Vector3f(pad, pad, pad);
	b.hi			= b.hi + Vector3f(pad, pad, pad);
	return b;
}

// appends a BLAS built over `tris` (already in the order of `boxes`); returns root node index
static uint32 appendBLAS(CompiledScene& s, const std::vector<prb_bvh_tri>& tris)
{
	BVHBuildInput in;
	in.boxes.resize(tris.size());
	for (size_t i = 0; i < tris.size(); ++i) {
		BoundingBox b;
		b.combine(Vector3f(tris[i].v0[0], tris[i].v0[1], tris[i].v0[2]));
		b.combine(Vector3f(tris[i].v1[0], tris[i].v1[1], tris[i].v1[2]));
		b.combine(Vector3f(tris[i].v2[0], tris[i].v2[1], tris[i].v2[2]));
		in.boxes[i] = padBox(b);
	}
	const BVH8 bvh		  = buildBVH8(in, 4);
	const uint32 nodeBase = (uint32)s.bvhNodes.size();
	const uint32 triBase  = (uint32)s.bvhTris.size();
	for (prb_bvh8_node n : bvh.nodes) {
		n.child_base += nodeBase;
		n.prim_base += triBase;
		s.bvhNodes.push_back(n);
	}
	for (uint32 p : bvh.primOrder)
		s.bvhTris.push_back(tris[p]);
	return nodeBase;
}

static prb_bvh_tri makeTri(const Vector3f& a, const Vector3f& b, const Vector3f& c, uint32 prim, uint32 flags)
{
	prb_bvh_tri t{};
	for (int i = 0; i < 3; ++i) {
		t.v0[i] = a[i];
		t.v1[i] = b[i];
		t.v2[i] = c[i];
	}
	t.prim_id = prim;
	t.flags	  = flags;
	return t;
}
// Embree quad (v0,v1,v2,v3) = triangles (v0,v1,v3) and (v2,v3,v1), second with u,v -> 1-u,1-v (SURVEY appendix B)
static void pushFaceTris(std::vector<prb_bvh_tri>& tris, const Vector3f& v0, const Vector3f& v1, const Vector3f& v2, const Vector3f* v3, uint32 prim)
{
	if (!v3) {
		tris.push_back(makeTri(v0, v1, v2, prim, 0));
	} else {
		tris.push_back(makeTri(v0, v1, *v3, prim, 0));
		tris.push_back(makeTri(v2, *v3, v1, prim, 1));
	}
}

uint32 SceneCompiler::registerMesh(const std::shared_ptr<MeshBase>& mesh)
{
	auto it = mMeshIDs.find(mesh.get());
	if (it != mMeshIDs.end())
		return it->second;
	CompiledScene& s = *mScene;
	prb_mesh m{};
	m.vertex_offset = (uint32)(s.vertices.size() / 3);
	m.vertex_count	= (uint32)mesh->vertexCount();
	m.face_offset	= (uint32)(s.faceIndices.size() / 4);
	m.face_count	= (uint32)mesh->faceCount();
	m.features		= (mesh->hasNormals() ? PRB_MESH_HAS_NORMALS : 0) | (mesh->hasUVs() ? PRB_MESH_HAS_UVS : 0);
	m.normal_offset = m.vertex_offset;
	m.uv_offset		= m.vertex_offset;
	s.vertices.insert(s.vertices.end(), mesh->vertices.begin(), mesh->vertices.end());
	if (mesh->hasNormals())
		s.normals.insert(s.normals.end(), mesh->normals.begin(), mesh->normals.end());
	else
		s.normals.resize(s.normals.size() + mesh->vertices.size(), 0.0f);
	if (mesh->hasUVs())
		s.uvs.insert(s.uvs.end(), mesh->uvs.begin(), mesh->uvs.end());
	else
		s.uvs.resize(s.uvs.size() + mesh->vertexCount() * 2, 0.0f);
	s.faceIndices.insert(s.faceIndices.end(), mesh->indices.begin(), mesh->indices.end());
	for (size_t f = 0; f < mesh->faceCount(); ++f)
		s.faceSlots.push_back(mesh->materialSlots.empty() ? 0 : mesh->materialSlots[f]);
	std::vector<prb_bvh_tri> tris;
	tris.reserve(mesh->faceCount());
	for (size_t f = 0; f < mesh->faceCount(); ++f) {
		const Vector3f v0 = mesh->vertex(mesh->indices[4 * f]), v1 = mesh->vertex(mesh->indices[4 * f + 1]), v2 = mesh->vertex(mesh->indices[4 * f + 2]);
		if (mesh->isQuad(f)) {
			const Vector3f v3 = mesh->vertex(mesh->indices[4 * f + 3]);
			pushFaceTris(tris, v0, v1, v2, &v3, (uint32)f);
		} else {
			pushFaceTris(tris, v0, v1, v2, nullptr, (uint32)f);
		}
	}
	m.blas_root = appendBLAS(s, tris);
	s.meshes.push_back(m);
	const uint32 id		= (uint32)s.meshes.size() - 1;
	mMeshIDs[mesh.get()] = id;
	return id;
}
uint32 SceneCompiler::registerEntityMaterials(const std::vector<uint32>& ids)
{
	const uint32 off = (uint32)mScene->entityMaterials.size();
	mScene->entityMaterials.insert(mScene->entityMaterials.end(), ids.begin(), ids.end());
	return off;
}

static void describeSamplers(Environment* env, CompiledScene& s)
{
	const RenderSettings& rs = env->renderSettings();
	const uint32 maxSamples	 = rs.maxSampleCount();
	// per-tile slot RNGs: Random(seed ^ (4201321 + slot)), slot AA=0, Lens=1, Time=2, Spectral=3 (RenderTile.cpp:10,33-35);
	// every tile constructs identical samplers from identical seeds, so one description serves all tiles.
	constexpr uint64 SLOT_RND_PRIME = 4201321;
	Random rAA(rs.seed ^ (SLOT_RND_PRIME + 0)), rLens(rs.seed ^ (SLOT_RND_PRIME + 1)), rTime(rs.seed ^ (SLOT_RND_PRIME + 2));
	rs.aaSamplerFactory->createInstance(maxSamples, rAA)->describe(s.desc.aa_sampler, s.pool);
	rs.lensSamplerFactory->createInstance(maxSamples, rLens)->describe(s.desc.lens_sampler, s.pool);
	rs.timeSamplerFactory->createInstance(maxSamples, rTime)->describe(s.desc.time_sampler, s.pool);
}

std::shared_ptr<CompiledScene> SceneCompiler::compile()
{
	mScene			 = std::make_shared<CompiledScene>();
	CompiledScene& s = *mScene;
	if (!mEnv->createDefaultsIfNecessary()) {
		PR_LOG(L_ERROR) << "Could not create default samplers/filter/mapper/integrator" << std::endl;
		return nullptr;
	}
	if (!mEnv->activeCamera) {
		PR_LOG(L_ERROR) << "No camera selected" << std::endl;
		return nullptr;
	}
	const RenderSettings& rs = mEnv->renderSettings();
	SceneDatabase& db		 = *mEnv->sceneDatabase();
	prb_settings& st		 = s.desc.settings;
	st.seed					 = rs.seed;
	st.film_width			 = rs.filmWidth;
	st.film_height			 = rs.filmHeight;
	st.view_x				 = rs.cropOffsetX();
	st.view_y				 = rs.cropOffsetY();
	st.view_w				 = rs.cropWidth();
	st.view_h				 = rs.cropHeight();
	st.max_sample_count		 = rs.maxSampleCount();
	st.spectral_mono		 = rs.spectralMono;
	st.film_monotonic		 = rs.spectralMono; // FrameOutputDevice(filter, viewSize, 3, spectralMono), loader/Environment.cpp:194-198
	st.want_variance		 = mEnv->outputSpecification().wantsVariance();
	st.want_aov_ext			 = mEnv->outputSpecification().wantsExtendedAOVs();
	st.spectral_hero		 = rs.spectralHero;
	st.spectral_start		 = rs.spectralStart;
	st.spectral_end			 = rs.spectralEnd;
	st.time_alpha			 = 1 * rs.timeScale; // TimeMappingMode::Right (RenderSettings.cpp:16, RenderTile.cpp:49-52)
	st.time_beta			 = 0;
	{
		const auto integrator = rs.integratorFactory->createInstance();
		integrator->describe(st);
		s.integrator = integrator->deviceIntegrator();
	}
	mEnv->activeCamera->describe(s.desc.camera);

	// spectral tables first in the pool
	s.desc.cie_offset = (uint32)s.pool.size();
	for (int c = 0; c < 3; ++c)
		s.pool.insert(s.pool.end(), CIE::table(c), CIE::table(c) + PR_CIE_SAMPLE_COUNT);

	NodeEmitter emitter;
	emitter.pool = &s.pool;
	for (const auto& m : db.Materials.getAll()) {
		prb_material pm{};
		for (auto& n : pm.node)
			n = PRB_INVALID_ID;
		m->describe(pm, emitter);
		s.materials.push_back(pm);
	}
	for (const auto& e : db.Emissions.getAll()) {
		prb_emission pe{};
		e->describe(pe, emitter);
		s.emissions.push_back(pe);
	}

	// entities + BLAS
	const auto t0 = std::chrono::steady_clock::now();
	BVHBuildInput tlasIn;
	for (const auto& e : db.Entities.getAll()) {
		prb_entity pe{};
		pe.emission_id = e->emissionID();
		pe.light_id	   = PRB_INVALID_ID;
		pe.visibility  = e->visibilityFlags();
		e->transform().to34(pe.local_to_world);
		e->invTransform().to34(pe.world_to_local);
		for (int i = 0; i < 9; ++i)
			pe.normal_matrix[i] = e->normalMatrix().m[i];
		pe.jacobian_det = e->volumeScalefactor();
		pe.world_area	= e->worldSurfaceArea();
		pe.pdf_area		= e->sampleParameterPointPDF();
		e->describe(pe, *this);
		if (pe.type == PRB_ENTITY_MESH) {
			pe.blas_root = s.meshes[pe.mesh_id].blas_root;
		} else if (pe.type == PRB_ENTITY_PLANE) {
			std::vector<prb_bvh_tri> tris;
			const float* q = &pe.geo[14];
			const Vector3f v0(q[0], q[1], q[2]), v1(q[3], q[4], q[5]), v2(q[6], q[7], q[8]), v3(q[9], q[10], q[11]);
			pushFaceTris(tris, v0, v1, v2, &v3, 0);
			pe.blas_root = appendBLAS(s, tris);
		} else {
			pe.blas_root = PRB_INVALID_ID;
		}
		const BoundingBox wb = e->worldBoundingBox();
		tlasIn.boxes.push_back(padBox(wb));
		s.sceneBounds.combine(wb);
		s.entities.push_back(pe);
	}
	{
		const BVH8 tlas		  = buildBVH8(tlasIn, 1);
		const uint32 nodeBase = (uint32)s.bvhNodes.size();
		for (prb_bvh8_node n : tlas.nodes) {
			n.child_base += nodeBase;
			s.bvhNodes.push_back(n);
		}
		s.tlasRefs		 = tlas.primOrder;
		s.desc.tlas_root = nodeBase;
	}
	s.bvhBuildSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();

	// origin-centred bounding sphere, Scene.cpp:106-120 (Sphere() starts with radius 1)
	s.sceneRadius = 1;
	if (s.sceneBounds.valid())
		s.sceneRadius = std::max(s.sceneRadius, std::max(s.sceneBounds.hi.norm(), s.sceneBounds.lo.norm()));

	// lights
	const SpectralRange cameraRange(rs.spectralStart, rs.spectralEnd);
	LightSampler ls(db, s.sceneRadius, cameraRange);
	for (const Light& l : ls.lights()) {
		prb_light pl{};
		pl.radiance_node = pl.background_node = PRB_INVALID_ID;
		if (l.isInfinite()) {
			l.infLight->describe(pl, emitter);
			pl.entity_id = pl.emission_id = PRB_INVALID_ID;
		} else {
			pl.type = PRB_LIGHT_AREA;
			const auto& ents = db.Entities.getAll();
			for (uint32 i = 0; i < ents.size(); ++i)
				if (ents[i].get() == l.entity)
					pl.entity_id = i;
			pl.emission_id					  = l.entity->emissionID();
			s.entities[pl.entity_id].light_id = l.id;
		}
		pl.select_pdf	= ls.selector().discretePdf(l.id);
		pl.scene_radius = s.sceneRadius;
		s.lights.push_back(pl);
	}
	s.lightCDF = ls.lights().empty() ? std::vector<float>{ 0.0f, 1.0f } : ls.selector().cdf();
	s.desc.inf_light_selection_probability = ls.infLightSelectionProbability();
	const SpectralRange lightRange		   = ls.lightSpectralRange();
	st.light_range_start				   = lightRange.Start;
	st.light_range_end					   = lightRange.End;

	// samplers, spectral mapper, filter
	describeSamplers(mEnv, s);
	SpectralMapperBuildInput smi;
	smi.cameraRange	 = cameraRange;
	smi.lightRange	 = lightRange;
	smi.lightSampler = &ls;
	rs.spectralMapperFactories.at("pixel")->describe(smi, s.desc.pixel_mapper, s.pool);
	{
		const auto filter = rs.pixelFilterFactory->createInstance();
		const int r		  = filter->radius();
		st.filter_radius  = r;
		st.filter_offset  = (uint32)s.pool.size();
		for (int y = -r; y <= r; ++y) // FilterCache, src/core/filter/FilterCache.h:6-31
			for (int x = -r; x <= r; ++x)
				s.pool.push_back(filter->evalWeight((float)x, (float)y));
	}
	// image textures evaluate SpectralUpsampler::prepare per lookup: the coefficient cube travels in the pool
	if (emitter.upsampler) {
		s.desc.upsampler_offset = (uint32)s.pool.size();
		s.desc.upsampler_res	= emitter.upsampler->resolution();
		s.pool.insert(s.pool.end(), emitter.upsampler->scale().begin(), emitter.upsampler->scale().end());
		s.pool.insert(s.pool.end(), emitter.upsampler->data().begin(), emitter.upsampler->data().end());
	}
	// light path expressions of the spectral output channels: dense DFA tables (lpe.cpp)
	for (const std::string& expr : mEnv->outputSpecification().lpeExpressions()) {
		const LPEAutomaton a = compileLPE(expr);
		if (!a.valid || a.stateCount > 255 || s.desc.n_lpe >= PRB_MAX_LPE) {
			PR_LOG(L_ERROR) << "Light path expression '" << expr << "' cannot be compiled for the device (" << a.stateCount << " states)" << std::endl;
			return nullptr;
		}
		prb_lpe& l	  = s.desc.lpe[s.desc.n_lpe++];
		l.n_states	  = a.stateCount;
		l.start_state = 0;
		l.next_offset = (uint32)s.lpeTables.size();
		s.lpeTables.insert(s.lpeTables.end(), a.next.begin(), a.next.end());
		l.final_offset = (uint32)s.lpeTables.size();
		s.lpeTables.insert(s.lpeTables.end(), a.final.begin(), a.final.end());
	}
	s.nodes = emitter.nodes;
	s.finalize();
	return mScene;
}

// ------------------------------------------------------------------ synthetic soup (SURVEY 8(d), C5)
namespace {
struct PCG32 { // pcg32 (XSH-RR 64/32) with the reference generator's default stream
	uint64 state, inc;
	explicit PCG32(uint64 seed, uint64 seq = 0xda3e39cb94b95bdbULL)
	{
		state = 0;
		inc	  = (seq << 1u) | 1u;
		next();
		state += seed;
		next();
	}
	uint32 next()
	{
		const uint64 old = state;
		state			 = old * 6364136223846793005ULL + inc;
		const uint32 xs	 = (uint32)(((old >> 18u) ^ old) >> 27u);
		const uint32 rot = (uint32)(old >> 59u);
		return (xs >> rot) | (xs << ((32 - rot) & 31));
	}
	float uniform() { return Random::uint32ToFloat(next()); }
};
} // namespace

std::shared_ptr<CompiledScene> makeSoupScene(uint32 triangles, uint64 seed, uint32 filmW, uint32 filmH)
{
	auto sp			 = std::make_shared<CompiledScene>();
	CompiledScene& s = *sp;
	PCG32 rng(seed);
	const float sz = 0.005f;
	s.vertices.resize((size_t)triangles * 9);
	s.faceIndices.resize((size_t)triangles * 4);
	s.faceSlots.assign(triangles, 0);
	std::vector<prb_bvh_tri> tris(triangles);
	for (uint32 t = 0; t < triangles; ++t) {
		float c[3];
		for (int k = 0; k < 3; ++k)
			c[k] = 2 * rng.uniform() - 1;
		Vector3f v[3];
		for (int j = 0; j < 3; ++j) {
			for (int k = 0; k < 3; ++k)
				v[j][k] = c[k] + sz * (2 * rng.uniform() - 1);
			for (int k = 0; k < 3; ++k)
				s.vertices[(size_t)t * 9 + j * 3 + k] = v[j][k];
			s.faceIndices[(size_t)t * 4 + j] = t * 3 + j;
		}
		s.faceIndices[(size_t)t * 4 + 3] = PRB_INVALID_ID;
		tris[t]							 = makeTri(v[0], v[1], v[2], t, 0);
	}
	s.normals.assign(s.vertices.size(), 0.0f);
	s.uvs.assign((size_t)triangles * 6, 0.0f);
	const auto t0 = std::chrono::steady_clock::now();
	prb_mesh m{};
	m.vertex_count = triangles * 3;
	m.face_count   = triangles;
	m.blas_root	   = appendBLAS(s, tris);
	s.meshes.push_back(m);
	prb_entity e{};
	e.type			  = PRB_ENTITY_MESH;
	e.mesh_id		  = 0;
	e.material_offset = 0;
	e.material_count  = 1;
	e.emission_id	  = PRB_INVALID_ID;
	e.light_id		  = PRB_INVALID_ID;
	e.visibility	  = 0x0F;
	e.blas_root		  = m.blas_root;
	Transformf::Identity().to34(e.local_to_world);
	Transformf::Identity().to34(e.world_to_local);
	for (int i = 0; i < 9; ++i)
		e.normal_matrix[i] = (i % 4 == 0) ? 1.0f : 0.0f;
	e.jacobian_det = 1;
	s.entities.push_back(e);
	s.entityMaterials.push_back(0);
	BVHBuildInput tl;
	BoundingBox wb;
	wb.combine(Vector3f(-1 - sz, -1 - sz, -1 - sz));
	wb.combine(Vector3f(1 + sz, 1 + sz, 1 + sz));
	tl.boxes.push_back(padBox(wb));
	s.sceneBounds = wb;
	{
		const BVH8 tlas		  = buildBVH8(tl, 1);
		const uint32 nodeBase = (uint32)s.bvhNodes.size();
		for (prb_bvh8_node n : tlas.nodes) {
			n.child_base += nodeBase;
			s.bvhNodes.push_back(n);
		}
		s.tlasRefs		 = tlas.primOrder;
		s.desc.tlas_root = nodeBase;
	}
	s.bvhBuildSeconds = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
	s.sceneRadius	  = std::max(1.0f, wb.hi.norm());
	// one white diffuse material, pinhole camera at (0,0,-3) looking +z, fov 40 deg
	prb_node cn{};
	cn.type = PRB_NODE_CONST;
	cn.p[0] = 0.8f;
	s.nodes.push_back(cn);
	prb_material mat{};
	mat.type	= PRB_MAT_DIFFUSE;
	mat.flags	= PRB_MATF_TWO_SIDED;
	mat.node[0] = 0;
	s.materials.push_back(mat);
	prb_settings& st	  = s.desc.settings;
	st.seed				  = 42;
	st.film_width		  = filmW;
	st.film_height		  = filmH;
	st.view_w			  = filmW;
	st.view_h			  = filmH;
	st.max_sample_count	  = 16;
	st.max_ray_depth	  = 2;
	st.soft_max_ray_depth = 2;
	st.do_nee = st.do_direct = st.emissive_scatter = 1;
	st.spectral_hero							   = 1;
	st.spectral_start							   = PR_CIE_WAVELENGTH_START;
	st.spectral_end								   = PR_CIE_WAVELENGTH_END;
	st.light_range_start						   = st.spectral_start;
	st.light_range_end							   = st.spectral_end;
	st.time_alpha								   = 1;
	const float half							   = std::tan(0.5f * 40.0f * PR_DEG2RAD);
	prb_camera& cam								   = s.desc.camera;
	cam.origin[2]								   = -3;
	cam.right[0]								   = half * (float)filmW / (float)filmH;
	cam.up[1]									   = half;
	cam.dir[2]									   = 1;
	cam.near_t									   = 1e-6f;
	cam.far_t									   = PR_INF;
	s.desc.aa_sampler.type = s.desc.lens_sampler.type = s.desc.time_sampler.type = PRB_SAMPLER_RANDOM;
	s.desc.aa_sampler.max_samples = s.desc.lens_sampler.max_samples = s.desc.time_sampler.max_samples = 16;
	s.desc.pixel_mapper.type													   = PRB_MAPPER_RANDOM;
	s.desc.cie_offset															   = 0;
	for (int c = 0; c < 3; ++c)
		s.pool.insert(s.pool.end(), CIE::table(c), CIE::table(c) + PR_CIE_SAMPLE_COUNT);
	st.filter_radius = 0;
	st.filter_offset = (uint32)s.pool.size();
	s.pool.push_back(1.0f);
	s.lightCDF = { 0.0f, 1.0f };
	s.finalize();
	return sp;
}
} // namespace PR
