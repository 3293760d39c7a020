/* prb200_abi.h -- the C ABI between PearRay-style C++17 host code and the B200 (sm_100a) CUDA
 * implementation of the spectral path-tracing hot path.
 *
 * Everything here is POD: plain pointers, sizes and integer status codes.  No C++ / torch types.
 * Host buffers are caller-owned; device memory is owned by the context.  One context per GPU,
 * used from one host thread (streams live inside the context).
 *
 * Each entry point names the reference interface (file:line under the PearRay checkout) it replaces.
 * All arithmetic is fp32 with FTZ/DAZ (reference src/base/Platform.h:20-34), ids are uint32.
 */
#ifndef PRB200_ABI_H
#define PRB200_ABI_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define PRB_ABI_VERSION 3u
#define PRB_INVALID_ID 0xFFFFFFFFu /* reference PR_INVALID_ID, src/base/config/Constants.inl */
#define PRB_SPECTRAL_BLOB_SIZE 4	/* reference SpectralBlob, src/core/spectral/SpectralBlob.h:7-20 */

typedef int32_t prb_status; /* 0 = ok, <0 = error; text via prb_last_error() */
#define PRB_OK 0
#define PRB_ERR_INVALID_ARG -1
#define PRB_ERR_CUDA -2
#define PRB_ERR_NO_SCENE -3
#define PRB_ERR_UNSUPPORTED -4
#define PRB_ERR_NO_DEVICE -5

/* ---------------------------------------------------------------- ray / hit streams */
/* Ray flags: reference RayFlag, src/core/ray/Ray.h:9-19 */
#define PRB_RAY_CAMERA 0x01u
#define PRB_RAY_LIGHT 0x02u
#define PRB_RAY_BOUNCE 0x04u
#define PRB_RAY_SHADOW 0x08u
#define PRB_RAY_MONOCHROME 0x10u

/* SoA ray stream as in reference RayStream (src/core/ray/RayStream.h:55-107): one array per
 * component.  Only the geometric part is needed by the trace entry points. */
typedef struct prb_ray_soa {
	const float* org_x;
	const float* org_y;
	const float* org_z;
	const float* dir_x;
	const float* dir_y;
	const float* dir_z;
	const float* tmin; /* may be NULL -> 1e-4 (BOUNCE_RAY_MIN, src/vcm/vcm/Defaults.h:4-7) */
	const float* tmax; /* may be NULL -> +inf */
} prb_ray_soa;

/* SoA hit stream as in reference HitStream / HitEntry (src/core/trace/HitEntry.h:7-15).  One entry
 * per ray, misses carry entity_id == PRB_INVALID_ID (reference Scene.cpp:185-189). */
typedef struct prb_hit_soa {
	uint32_t* entity_id;
	uint32_t* primitive_id;
	float* u;
	float* v;
	float* t;
} prb_hit_soa;

/* ---------------------------------------------------------------- shading nodes */
/* Flattened shading network (reference FloatSpectralNode graph, src/core/shader/INode.h). */
enum {
	PRB_NODE_CONST		  = 0, /* p[0]                       ConstSpectralNode, loader/shader/ConstNode.cpp:27-36 */
	PRB_NODE_PARAM		  = 1, /* p[0..2] = a,b,c            ParametricSpectralNode :59-62 ('refl') */
	PRB_NODE_PARAM_SCALED = 2, /* p[0..2], p[3] = power      ParametricScaledSpectralNode :85-88 ('illum') */
	PRB_NODE_TABLE		  = 3, /* a=pool offset,b=count,p[0]=start nm,p[1]=end nm   EquidistantSpectrumView::lookup */
	PRB_NODE_SELLMEIER	  = 4, /* a=pool offset (B[n],C[n]), b=n   SellmeierIndexNode, node/ReflectiveNode.cpp:104-140 */
	PRB_NODE_MUL		  = 5, /* a,b = node ids             MulSpectralMath ('smul') */
	PRB_NODE_CHECKER	  = 6, /* a,b = node ids, p[0]=su,p[1]=sv,p[2]=mode(0 none,1 iso,2 aniso)  CheckerboardNode.cpp:26-48 */
	/* NonParametricImageNode (loader/shader/ImageNode.cpp:93-162): a = pool offset of width*height RGB texels (rows top to
	 * bottom as stored in the file), b = width | height << 16, p[0] = interpolation (PRB_TEX_*), p[1] / p[2] = wrap mode of
	 * s / t (PRB_WRAP_*), p[3] != 0: the file is sRGB encoded -> RGBConverter::linearize after the lookup.  The texel fetch
	 * restates OpenImageIO's TextureSystem::texture() without MIP levels and derivatives (an un-vendored dependency of the
	 * reference: texel centres at (i + 0.5) / size, t = 1 - v), then SpectralUpsampler::prepare + ::compute per lookup
	 * against the coefficient cube at prb_scene_desc::upsampler_offset. */
	PRB_NODE_IMAGE = 7
};
enum { PRB_TEX_CLOSEST = 0, PRB_TEX_BILINEAR = 1, PRB_TEX_BICUBIC = 2 };
enum { PRB_WRAP_BLACK = 0, PRB_WRAP_CLAMP = 1, PRB_WRAP_PERIODIC = 2, PRB_WRAP_MIRROR = 3 };
#define PRB_NODE_FLAG_SPECTRAL_VARYING 0x1u /* NodeFlag::SpectralVarying */
#define PRB_NODE_FLAG_TEXTURE_VARYING 0x2u

typedef struct prb_node {
	uint32_t type;
	uint32_t flags;
	uint32_t a;
	uint32_t b;
	float p[4];
} prb_node;

/* ---------------------------------------------------------------- materials */
enum {
	PRB_MAT_DIFFUSE			= 0, /* plugins/main/materials/lambert.cpp:14-89        node[0]=albedo */
	PRB_MAT_DIELECTRIC		= 1, /* dielectric.cpp:18-135   node[0]=specularity node[1]=transmission node[2]=ior */
	PRB_MAT_CONDUCTOR		= 2, /* conductor.cpp:16-95     node[0]=eta node[1]=k node[2]=specularity */
	PRB_MAT_ROUGHCONDUCTOR	= 3, /* roughconductor.cpp:16-143  nodes as CONDUCTOR, f[0]=roughness_x f[1]=roughness_y */
	PRB_MAT_ROUGHDIELECTRIC = 4, /* roughdielectric.cpp:42-279 nodes as DIELECTRIC, f[0],f[1] roughness */
	PRB_MAT_PRINCIPLED		= 5, /* principled.cpp:34-631   node[0]=base node[1]=ior, f[] see PRB_PR_* */
	PRB_MAT_MIRROR			= 6, /* mirror.cpp:14-65        node[0]=specularity (only-delta) */
	PRB_MAT_ORENNAYAR		= 7, /* orennayar.cpp:16-86     node[0]=albedo, f[0]=roughness (scalar, squared on use) */
	/* blend.cpp:20-148 / add.cpp:20-122: node[0], node[1] = MATERIAL ids of the two children (leaf materials only, no nesting
	 * on the device path), f[0] = blend factor; PRB_MATF_CHILD0_DELTA / CHILD1_DELTA give the MaterialDelta variant */
	PRB_MAT_BLEND = 8,
	PRB_MAT_ADD	  = 9
};
#define PRB_MATF_TWO_SIDED 0x001u		  /* lambert two_sided (default true) */
#define PRB_MATF_THIN 0x002u			  /* dielectric / principled 'thin' */
#define PRB_MATF_TRANSMISSION_COLOR 0x004u /* dielectric 'transmission' given */
#define PRB_MATF_VNDF 0x008u			  /* rough*: 'vndf' (default true) */
#define PRB_MATF_ANISOTROPIC 0x010u		  /* rough*: roughness_x != roughness_y node */
#define PRB_MATF_ONLY_DELTA 0x020u		  /* IMaterial::hasOnlyDeltaDistribution() */
#define PRB_MATF_SPECTRAL_VARYING 0x040u  /* mNodeContribFlags & SpectralVarying (hero collapse when delta) */
#define PRB_MATF_HAS_TRANSMISSION 0x080u  /* principled: diffuse_/specular_transmission present */
#define PRB_MATF_CHILD0_DELTA 0x100u	  /* blend / add: material1 has only delta distributions */
#define PRB_MATF_CHILD1_DELTA 0x200u	  /* blend / add: material2 has only delta distributions */

/* principled scalar slots (principled.cpp:50-62) */
enum {
	PRB_PR_DIFF_TRANS = 0,
	PRB_PR_ROUGHNESS,
	PRB_PR_ANISOTROPIC,
	PRB_PR_SPEC_TRANS,
	PRB_PR_SPEC_TINT,
	PRB_PR_FLATNESS,
	PRB_PR_METALLIC,
	PRB_PR_SHEEN,
	PRB_PR_SHEEN_TINT,
	PRB_PR_CLEARCOAT,
	PRB_PR_CLEARCOAT_GLOSS,
	PRB_PR__COUNT
};

typedef struct prb_material {
	uint32_t type;
	uint32_t flags;
	uint32_t node[4];
	float f[12];
} prb_material;

typedef struct prb_emission { /* plugins/main/emissions/diffuse.cpp:11-56 */
	uint32_t radiance_node;
	uint32_t _pad;
} prb_emission;

/* ---------------------------------------------------------------- geometry */
enum {
	PRB_ENTITY_MESH	  = 0, /* plugins/main/entities/mesh.cpp   (instance of a mesh BLAS) */
	PRB_ENTITY_SPHERE = 1, /* sphere.cpp  (RTC_GEOMETRY_TYPE_SPHERE_POINT) */
	PRB_ENTITY_PLANE  = 2  /* plane.cpp   (one world-space quad) */
};
#define PRB_MESH_HAS_NORMALS 0x1u
#define PRB_MESH_HAS_UVS 0x2u

/* Mesh data lives in shared pools (scene.vertices / normals / uvs / face_indices / face_slots).
 * Faces are stored as 4 indices; triangles carry PRB_INVALID_ID in the 4th (reference mixed
 * index layout, mesh.cpp:30-46).  Index values are relative to the mesh's vertex_offset. */
typedef struct prb_mesh {
	uint32_t vertex_offset; /* in vertices (x3 floats) */
	uint32_t vertex_count;
	uint32_t face_offset; /* in faces */
	uint32_t face_count;
	uint32_t features;
	uint32_t blas_root;		 /* node index of the mesh BVH root inside scene.bvh_nodes */
	uint32_t uv_offset;		 /* in uvs (x2 floats); one per vertex when HAS_UVS */
	uint32_t normal_offset;	 /* in normals (x3 floats); one per vertex when HAS_NORMALS */
} prb_mesh;

/* geo[] layout
 *  SPHERE: [0..2] world centre, [3] world radius (radius * mean column norm, sphere.cpp:91-100),
 *          [4] local radius, [5] 1/worldSurfaceArea (mPDF_Cache, sphere.cpp:31)
 *  PLANE : [0..2] mS, [3..5] mEx, [6..8] mEy, [9..11] mEz (unit), [12] width, [13] height
 *          (plane.cpp:227-244), [14..25] the four world-space quad corners p, p+y, p+y+x, p+x
 *          (plane.cpp:80-84), [26..28] normalMatrix*plane.normal (un-normalised, plane.cpp:175),
 *          [29..31] local plane position, [32..34] local x axis, [35..37] local y axis,
 *          [38] 1/|x|^2, [39] 1/|y|^2 (Plane::project, src/core/geometry/Plane.cpp:117-123)
 *  MESH  : unused */
typedef struct prb_entity {
	uint32_t type;
	uint32_t mesh_id;
	uint32_t material_offset; /* into scene.entity_materials; mesh: per slot, sphere/plane: one */
	uint32_t material_count;
	uint32_t emission_id;
	uint32_t light_id; /* index into scene.lights or PRB_INVALID_ID */
	uint32_t visibility; /* EntityVisibility bits == ray flags, src/core/entity/IEntity.h:9-15 */
	uint32_t blas_root;
	float local_to_world[12]; /* row-major 3x4, ITransformable::transform() */
	float world_to_local[12]; /* invTransform() */
	float normal_matrix[9];	  /* row-major 3x3, linear().inverse().transpose() */
	float jacobian_det;		  /* volumeScalefactor(), ITransformable.cpp:14 */
	float world_area;		  /* IEntity::worldSurfaceArea() */
	float pdf_area;			  /* sampleParameterPointPDF() without info */
	float geo[45];
} prb_entity;

/* BVH8 compressed node, 80 bytes (host builder: pearray_b200/host/bvh_builder.cpp).
 * child boxes: lo = p + q_lo * 2^e, hi = p + q_hi * 2^e per axis.
 * meta[i]: 0xFF empty; 0x80|k internal child, node index = child_base + k;
 *          otherwise leaf: ((count-1) << 5) | offset, prims [prim_base+offset, +count), count<=4. */
typedef struct prb_bvh8_node {
	float px, py, pz;
	uint8_t ex, ey, ez, imask;
	uint32_t child_base;
	uint32_t prim_base;
	uint8_t meta[8];
	uint8_t qlo_x[8], qlo_y[8], qlo_z[8];
	uint8_t qhi_x[8], qhi_y[8], qhi_z[8];
} prb_bvh8_node;

/* 48-byte leaf primitive: a triangle.  prim_id = face index in its mesh (0 for planes);
 * flags bit0: second triangle of a quad (u,v -> 1-u,1-v; Embree quad convention, SURVEY App. B). */
typedef struct prb_bvh_tri {
	float v0[3];
	uint32_t prim_id;
	float v1[3];
	uint32_t flags;
	float v2[3];
	uint32_t _pad;
} prb_bvh_tri;

/* ---------------------------------------------------------------- lights */
enum {
	PRB_LIGHT_AREA		= 0,
	PRB_LIGHT_ENV		= 1, /* plugins/main/infinitelights/environment.cpp; dist_w > 0: the Distribution2D branches (image based radiance) */
	PRB_LIGHT_SKY		= 2, /* plugins/main/infinitelights/sky.cpp:27-173 (Hosek-Wilkie table + Distribution2D) */
	PRB_LIGHT_SUN		= 3, /* plugins/main/infinitelights/sun.cpp:27-140 (cone) */
	PRB_LIGHT_SUN_DELTA = 4	 /* plugins/main/infinitelights/sun.cpp:142-240 (radius <= eps: delta direction) */
};
#define PRB_SKY_BANDS 11		 /* AR_SPECTRAL_BANDS, src/skysun/skysun/SkySunConfig.h:6-9 */
#define PRB_SKY_BAND_START 320.0f /* AR_SPECTRAL_START */
#define PRB_SKY_BAND_DELTA 40.0f	 /* AR_SPECTRAL_DELTA */
typedef struct prb_light { /* src/core/light/Light.cpp, LightSampler.cpp:11-132 */
	uint32_t type;
	uint32_t entity_id;	   /* AREA */
	uint32_t emission_id;  /* AREA */
	uint32_t radiance_node; /* ENV: radiance;  (environment.cpp) */
	uint32_t background_node; /* ENV: background (used at depth 0 when split) */
	uint32_t env_split;
	float select_pdf; /* discretePdf(lightID) */
	float scene_radius;
	float normal_matrix[9];		/* ENV/SKY: ITransformable normalMatrix() */
	float inv_normal_matrix[9]; /* ENV/SKY: invNormalMatrix() */
	/* SKY: SkyModel::mData [elevation][azimuth][PRB_SKY_BANDS] floats at table_offset in the pool (SkyModel.cpp:19-60);
	 * SUN / SUN_DELTA: the EquidistantSpectrum (table_count samples over [table_start, table_end] nm) */
	uint32_t table_offset;
	uint32_t table_count;
	float table_start, table_end;
	uint32_t az_count, el_count; /* SKY */
	/* SKY: Distribution2D (core/sampler/Distribution2D.cpp) at dist_offset in the pool: marginal CDF (dist_h + 1 floats)
	 * followed by dist_h conditional CDFs of (dist_w + 1) floats each */
	uint32_t dist_offset, dist_w, dist_h;
	uint32_t sky_extend; /* SkyLight<ExtendToGround> */
	float sun_dir[3], sun_dx[3], sun_dy[3]; /* SUN: mDirection and its tangent frame */
	float sun_cos_theta, sun_pdf;			 /* SUN: cos(SUN_VIS_RADIUS * radius), uniform_cone_pdf */
} prb_light;

/* ---------------------------------------------------------------- samplers, mapper, camera */
enum {
	PRB_SAMPLER_RANDOM	   = 0,
	PRB_SAMPLER_MJITT	   = 1,
	PRB_SAMPLER_SOBOL	   = 2,
	PRB_SAMPLER_STRATIFIED = 3, /* StratifiedSampler.cpp:12-41: bins_1d = groups, m2d_x = (uint32)sqrt(groups) */
	PRB_SAMPLER_UNIFORM	   = 4, /* UniformSampler.cpp:11-29: always 0.5 */
	/* HaltonSampler.cpp:14-121 (halton and hammersley): tables like SOBOL at table_offset; past max_samples the radical
	 * inverse of (index + seed) in base m2d_x (x) / m2d_y (y; 47 for hammersley) is computed on the fly; seed = burn-in */
	PRB_SAMPLER_HALTON	   = 5
};
typedef struct prb_sampler { /* src/plugins/main/sampler/ */
	uint32_t type;
	uint32_t max_samples; /* ISampler::maxSamples() */
	uint32_t bins_1d;	  /* mjitt m1D */
	uint32_t m2d_x, m2d_y;
	uint32_t seed;			/* mjitt mSeed */
	uint32_t table_offset;	/* sobol: pool offset of max_samples 1D floats followed by max_samples (x,y) pairs */
	uint32_t _pad;
} prb_sampler;

enum {
	PRB_MAPPER_RANDOM	= 0,
	PRB_MAPPER_SPD_CMIS = 1,
	PRB_MAPPER_SPD_HERO = 2,
	PRB_MAPPER_CIE		= 3, /* cie.cpp:13-83: four independent samples of the CIE Y or X+Y+Z CDF, truncated to the camera range */
	/* agh.cpp:14-121 ("An Improved Technique for Full Spectral Rendering"): lambda = B - atanh(C - N u) / A with A = 0.0072,
	 * B = 538; trunc_cdf_start holds C = tanh(A (B - start)), trunc_cdf_end holds N = C - tanh(A (B - end)) */
	PRB_MAPPER_AGH_CMIS = 4, /* four independent samples */
	PRB_MAPPER_AGH_HERO = 5	 /* one sample + hero rotation (Standard.h:8-21) */
};
typedef struct prb_spectral_mapper { /* src/plugins/main/spectralmapper/spd.cpp, random.cpp, cie.cpp */
	uint32_t type;
	uint32_t cdf_offset; /* pool offset of cdf_size floats (Distribution1D mCDF / StaticCDF) */
	uint32_t cdf_size;
	/* CIE: evalContinuous of the CDF at the normalised ends of the camera range (CIE::sample_trunc, CIE.h:117-127);
	 * 0 and 1 for the full range */
	float trunc_cdf_start, trunc_cdf_end;
} prb_spectral_mapper;

enum {
	PRB_CAMERA_PERSPECTIVE	= 0, /* plugins/main/cameras/perspective.cpp:45-113, no-DOF branch: origin fixed, dir = normalize(right nx + up ny + dir) */
	PRB_CAMERA_ORTHOGRAPHIC = 1	 /* plugins/main/cameras/ortho.cpp:47-66: origin + right nx + up ny, dir = mDirection_Cache (unit) */
};
typedef struct prb_camera {
	float origin[3];
	float right[3]; /* mRight_Cache (already * 0.5 * width) */
	float up[3];	/* mUp_Cache */
	float dir[3];	/* perspective: mFocalDistance_Cache; orthographic: mDirection_Cache (normalised) */
	float near_t, far_t;
	uint32_t type; /* PRB_CAMERA_* */
	uint32_t has_dof; /* PerspectiveCamera<HasDOF = true> (perspective.cpp:66-75): the lens sample moves the origin inside the aperture */
	float aperture_x[3]; /* mXApertureRadius_Cache */
	float aperture_y[3]; /* mYApertureRadius_Cache */
} prb_camera;

typedef struct prb_settings { /* RenderSettings.cpp:11-33 + DiParameters direct.cpp:34-39 */
	uint64_t seed;
	uint32_t film_width, film_height;
	uint32_t view_x, view_y, view_w, view_h; /* crop window in film pixels */
	uint32_t max_sample_count;				 /* RenderSettings::maxSampleCount() */
	uint32_t max_ray_depth;					 /* hard, default 64 */
	uint32_t soft_max_ray_depth;			 /* default 4 */
	uint32_t mis_power;						 /* 0 balance, 1 power */
	uint32_t do_nee, do_direct, emissive_scatter;
	uint32_t spectral_mono, spectral_hero;
	float spectral_start, spectral_end; /* camera range */
	float light_range_start, light_range_end;
	float time_alpha, time_beta; /* RenderTile.cpp:44-63 */
	int32_t filter_radius;		 /* FilterCache table (2r+1)^2 at filter_offset in the pool */
	uint32_t filter_offset;
	/* monotonic film: FrameOutputDevice(filter, size, 3, spectralMono) (loader/Environment.cpp:194-198) -> every fragment
	 * stores its unweighted hero sample in all three channels (mapSpectral<true>, LocalFrameOutputDevice.cpp:76-85) */
	uint32_t film_monotonic;
	/* accumulate AOV_OnlineMean / AOV_OnlineVariance (src/core/buffer/VarianceEstimator.inl:16-28, driven per merged tile and
	 * iteration from FrameOutputDevice::mergeLocal, loader/output/FrameOutputDevice.cpp:104-109): set by the host when an
	 * (output ...) block asks for a `variance` / `online_mean` channel */
	uint32_t want_variance;
	/* accumulate the extended shading-point AOVs of prb_film_download_aov_ext (tangent, bitangent, view, material / emission id):
	 * set by the host when an (output ...) block asks for one of them */
	uint32_t want_aov_ext;
} prb_settings;

/* ---------------------------------------------------------------- light path expressions
 * One compiled `:lpe` expression of an (output (channel ...)) block (reference src/core/path/LightPathExpression.cpp,
 * LPE_Automaton.cpp): a dense DFA over the 15 path-token symbols  symbol = ScatteringType * 3 + ScatteringEvent
 * (LightPathToken.h:6-20: Camera, Emissive, Refraction, Reflection, Background x Diffuse, Specular, None).
 * next[state * 15 + symbol] is the next state or PRB_LPE_REJECT; final[state] != 0 marks accepting states.  A fragment is
 * added to the channel when the automaton, started in start_state, accepts the fragment's token string
 * (LocalFrameOutputDevice.cpp:100-111). */
#define PRB_MAX_LPE 8u
#define PRB_LPE_SYMBOLS 15u
#define PRB_LPE_REJECT 0xFFu
typedef struct prb_lpe {
	uint32_t next_offset;  /* into prb_scene_desc::lpe_tables: n_states * 15 bytes */
	uint32_t final_offset; /* into lpe_tables: n_states bytes */
	uint32_t n_states;	   /* <= 255 */
	uint32_t start_state;
} prb_lpe;

/* ---------------------------------------------------------------- the scene */
typedef struct prb_scene_desc {
	uint32_t abi_version;
	prb_settings settings;
	prb_camera camera;
	prb_sampler aa_sampler, lens_sampler, time_sampler;
	prb_spectral_mapper pixel_mapper;

	uint32_t n_nodes;
	const prb_node* nodes;
	uint32_t n_materials;
	const prb_material* materials;
	uint32_t n_emissions;
	const prb_emission* emissions;
	uint32_t n_entities;
	const prb_entity* entities;
	uint32_t n_entity_materials;
	const uint32_t* entity_materials;
	uint32_t n_meshes;
	const prb_mesh* meshes;
	uint32_t n_vertices;
	const float* vertices; /* xyz */
	const float* normals;  /* xyz per vertex (0 when mesh has none) */
	const float* uvs;	   /* uv per vertex */
	uint32_t n_faces;
	const uint32_t* face_indices; /* 4 per face */
	const uint32_t* face_slots;	  /* material slot per face */

	uint32_t n_lights;
	const prb_light* lights;
	const float* light_cdf; /* n_lights + 1 */
	float inf_light_selection_probability;

	uint32_t tlas_root; /* node index */
	uint32_t n_bvh_nodes;
	const prb_bvh8_node* bvh_nodes;
	uint32_t n_bvh_tris;
	const prb_bvh_tri* bvh_tris;
	uint32_t n_tlas_refs;
	const uint32_t* tlas_refs; /* TLAS leaf prim -> entity id */

	uint32_t n_pool;
	const float* pool; /* CIE tables, illuminants, CDFs, Sobol tables, filter table */
	uint32_t cie_offset; /* 3 x 441 floats: x, y, z (CIE 2006, 390..830 nm) */
	uint32_t _pad;

	/* RGB -> spectrum coefficient cube of the SpectralUpsampler (src/core/spectral/SpectralUpsampler.cpp; Jakob & Hanika 2019)
	 * for image textures, in the pool: upsampler_res scale values, then 3 * res^3 * 3 coefficients; 0 / 0 when the scene has
	 * no image node */
	uint32_t upsampler_offset, upsampler_res;
	/* spectral output channels restricted by a light path expression (at most PRB_MAX_LPE) */
	uint32_t n_lpe;
	uint32_t n_lpe_bytes;
	const uint8_t* lpe_tables;
	prb_lpe lpe[PRB_MAX_LPE];
} prb_scene_desc;

/* One render tile (reference RenderTile start/end, src/core/renderer/RenderTile.h).  Pixels are film
 * coordinates; [sx,ex) x [sy,ey). */
typedef struct prb_tile {
	uint32_t sx, sy, ex, ey;
} prb_tile;

/* reference RenderStatisticEntry, src/core/renderer/RenderStatistics.h:9-24 */
typedef struct prb_stats {
	uint64_t camera_ray_count, light_ray_count, primary_ray_count, bounce_ray_count, shadow_ray_count,
		monochrome_ray_count, pixel_sample_count, entity_hit_count, background_hit_count,
		camera_depth_count, light_depth_count;
	uint64_t kernel_launches; /* CUDA kernels launched by this context so far */
	uint64_t wavefront_iterations;
} prb_stats;

/* material unit-call contexts: reference MaterialEvalContext / MaterialSampleContext
 * (src/core/material/MaterialContext.h:12-110), all in shading space (N = +z) */
typedef struct prb_material_query {
	float V[3];
	float L[3]; /* eval / pdf only */
	float wavelength_nm[4];
	float uv[2];
	uint32_t ray_flags;
	uint32_t material_id;
	uint64_t rng_state; /* sample only: pcg32_fast state; updated state is returned */
} prb_material_query;

typedef struct prb_material_result {
	float weight[4]; /* eval: Weight; sample: IntegralWeight */
	float pdf_s[4];
	float L[3]; /* sample only */
	uint32_t flags; /* MaterialSampleFlag bits, src/core/material/MaterialType.h */
	uint32_t type;	/* MaterialScatteringType */
	uint64_t rng_state;
} prb_material_result;

typedef struct prb_ctx prb_ctx;

/* -- life cycle.  Replaces RenderFactory::create / RenderContext ctor (src/core/renderer/RenderFactory.cpp:16-42). */
prb_status prb_create(int device, prb_ctx** out);
void prb_destroy(prb_ctx* ctx);
const char* prb_last_error(void);
int prb_device_count(void);

/* -- scene upload.  Replaces Scene::setupScene + rtcCommitScene (src/core/scene/Scene.cpp:88-120):
 * the BVH is built by the host (SAH BVH8) and arrives inside the descriptor. */
prb_status prb_upload_scene(prb_ctx* ctx, const prb_scene_desc* scene);

/* -- per-film-pixel RNG states.  Replaces RenderRandomMap (src/core/renderer/RenderRandomMap.cpp:11-28);
 * n must be film_width*film_height. */
prb_status prb_upload_rng(prb_ctx* ctx, const uint64_t* states, size_t n);
prb_status prb_download_rng(prb_ctx* ctx, uint64_t* states, size_t n);

/* -- the hot path.  Replaces IIntegratorInstance::onTile for the 'direct' integrator
 * (src/plugins/main/integrators/direct.cpp:153-166) over a batch of tiles, for iterations
 * [first_iteration, first_iteration + iteration_count).  Film cells of the tiles are updated
 * (running mean over iterations as FrameOutputDevice::onEndOfIteration, FrameOutputDevice.cpp:202-221).
 * Blocks until every sample of the call has been folded into the film (the wavefront loop polls a device counter).
 * first_iteration == 0 starts the listed pixels from scratch (sample counts, AOV sums and feedback bits are cleared);
 * tiles must not overlap; prb_upload_rng must have been called since the last prb_upload_scene. */
prb_status prb_render_tiles(prb_ctx* ctx, const prb_tile* tiles, size_t n_tiles,
							uint32_t first_iteration, uint32_t iteration_count);
prb_status prb_sync(prb_ctx* ctx);
prb_status prb_film_clear(prb_ctx* ctx);

/* -- film read-back.  Replaces FrameOutputDevice / FrameContainer channel access
 * (src/loader/output/FrameOutputDevice.cpp).  xyz: W*H*3 floats (pixel filter applied),
 * sample_count: W*H (AOV_SampleCount).  Either may be NULL. */
prb_status prb_film_download(prb_ctx* ctx, float* xyz, uint32_t* sample_count);
/* optional first-hit AOVs (sums over samples as commitShadingPoints, LocalFrameOutputDevice.cpp:252-302):
 * normal (3), position (3), uv (2), depth (1), entity id (1) -> 10 floats per pixel, may be NULL */
prb_status prb_film_download_aov(prb_ctx* ctx, float* aov10);
/* the remaining shading-point AOVs of commitShadingPoints (LocalFrameOutputDevice.cpp:268-284), sums over the samples,
 * PRB_AOV_EXT floats per pixel: tangent Nx (3), bitangent Ny (3), view direction (3), material id, emission id.
 * (AOV_NormalG equals AOV_Normal on this path -- IntersectionPoint::setForSurface copies Geometry.N -- and AOV_DisplaceID is
 * PR_INVALID_ID for every entity type of the path; both are produced by the host writer.) */
#define PRB_AOV_EXT 11u
prb_status prb_film_download_aov_ext(prb_ctx* ctx, float* aov11);
/* AOV_Feedback (LocalFrameOutputDevice.cpp:125-143, FrameOutputDevice.cpp:150-153): per pixel the OR of the PRB_FEEDBACK_*
 * bits of every fragment that was rejected there; W*H words */
#define PRB_FEEDBACK_NAN 0x1u		/* OutputFeedback::NaN, src/core/output/Feedback.h:6-12 */
#define PRB_FEEDBACK_INFINITE 0x2u	/* OutputFeedback::Infinite */
#define PRB_FEEDBACK_NEGATIVE 0x4u	/* OutputFeedback::Negative */
prb_status prb_film_download_feedback(prb_ctx* ctx, uint32_t* feedback);
/* AOV_OnlineMean and AOV_OnlineVariance of the unfiltered per-iteration pixel value (W*H*3 floats each; either may be NULL):
 * Welford's update exactly as VarianceEstimator::addValue writes it.  Identical to the reference for a radius-0 pixel filter
 * (the reference feeds the estimator the FILTERED tile image of every iteration, and pixels under the filter footprint of
 * two tiles twice per iteration in thread order -- not reproducible even by the reference itself).  PRB_ERR_UNSUPPORTED unless
 * prb_settings.want_variance was set at upload. */
prb_status prb_film_download_variance(prb_ctx* ctx, float* online_mean, float* online_variance);
/* the spectral channel of light path expression `index` (prb_scene_desc::lpe): XYZ running mean of the fragments whose path the
 * expression accepts, 3 floats per film pixel, pixel filter applied like prb_film_download
 * (LocalFrameOutputDevice.cpp:100-111, FrameOutputDevice.cpp:216-218) */
prb_status prb_film_download_lpe(prb_ctx* ctx, uint32_t index, float* xyz);
/* copy the UNFILTERED film (xyz mean, 3 floats/pixel, then sample counts as float) into a caller
 * provided DEVICE buffer of W*H*4 floats -- the buffer handed to the NCCL reduce in multi-GPU runs. */
prb_status prb_film_export_device(prb_ctx* ctx, float* device_dst);
/* load an (already reduced) unfiltered film back and apply the pixel filter */
prb_status prb_film_import_device(prb_ctx* ctx, const float* device_src);

/* -- multi-GPU film combine (SURVEY 8(e); replaces the image-tile contexts of RenderFactory::create,
 * src/core/renderer/RenderFactory.cpp:16-42, whose per-context outputs the reference client merges on the host,
 * src/client/main.cpp:172-173).  The scene is replicated; every context renders its share and ONE reduction of the
 * UNFILTERED film (xyz running mean + sample count + the ten AOV sums + feedback bits) lands in the root context, which
 * then serves prb_film_download (pixel filter applied after the reduce).
 *   PRB_PARTITION_TILES    every film pixel was rendered by exactly one context (interleaved tiles): plain sum, the
 *                          root film is bit-identical to a single-context render of the same tiles
 *   PRB_PARTITION_SAMPLES  every context rendered the whole film for its own iteration range [first, end) starting from
 *                          an empty film (so its mean is sum / end): contexts are weighted end_r / total_iterations with
 *                          total_iterations = the sum of the range lengths, counts / AOV sums / feedback bits add up */
#define PRB_PARTITION_TILES 0
#define PRB_PARTITION_SAMPLES 1
/* one process driving several GPUs: ctxs[0] is the root.  With peer access the root reads the other films directly over
 * NVLink inside ONE kernel (sum + import, no staging copy); without it the films are staged with cudaMemcpyPeer. */
prb_status prb_film_reduce(prb_ctx** ctxs, int n_ctx, int partition);
/* one process per GPU (torchrun / MPI): NCCL.  Rank 0 calls prb_comm_unique_id and ships the 128 bytes to the other ranks
 * out of band (torch.distributed store, MPI_Bcast, a file ...); every rank calls prb_comm_init, then prb_film_reduce_comm
 * once per render (collective: ncclReduce over NVLink on the context stream, root imports).  libnccl.so.2 is loaded at run
 * time (the copy already in the process, e.g. torch's, else the system one): PRB_ERR_UNSUPPORTED when there is none. */
#define PRB_COMM_UNIQUE_ID_BYTES 128
prb_status prb_comm_unique_id(uint8_t id[PRB_COMM_UNIQUE_ID_BYTES]);
prb_status prb_comm_init(prb_ctx* ctx, const uint8_t id[PRB_COMM_UNIQUE_ID_BYTES], int rank, int world);
prb_status prb_comm_destroy(prb_ctx* ctx);
prb_status prb_film_reduce_comm(prb_ctx* ctx, int partition, uint32_t total_iterations, int root);
/* device ms (CUDA events on the context stream) of the last prb_film_reduce / prb_film_reduce_comm of this context */
prb_status prb_last_reduce_ms(prb_ctx* ctx, float* ms);

/* -- stream tracing.  Replace Scene::traceRays (Scene.cpp:138-218, rtcIntersect16) and
 * Scene::traceShadowRay (Scene.cpp:266-280, rtcOccluded1; occluded[i] = 1 if anything was hit in
 * [tmin, tmax]).  Host-pointer variants copy in/out (page-locked host columns are copied at link speed: 467 M rays/s end to end
 * on the 10 M-triangle soup against 96 M from pageable arrays); *_device variants take device pointers. */
prb_status prb_trace_closest(prb_ctx* ctx, const prb_ray_soa* rays, size_t n, prb_hit_soa* hits);
prb_status prb_trace_any(prb_ctx* ctx, const prb_ray_soa* rays, size_t n, uint8_t* occluded);
prb_status prb_trace_closest_device(prb_ctx* ctx, const prb_ray_soa* rays, size_t n, prb_hit_soa* hits);
prb_status prb_trace_any_device(prb_ctx* ctx, const prb_ray_soa* rays, size_t n, uint8_t* occluded);
/* camera rays of one iteration for the given tiles (RenderTile::constructCameraRay, RenderTile.cpp:71-132)
 * written as a host SoA stream; does not advance the context's RNG states. n_out receives the count. */
prb_status prb_generate_camera_rays(prb_ctx* ctx, const prb_tile* tiles, size_t n_tiles, uint32_t iteration,
									float* org_xyz, float* dir_xyz, float* wavelengths4, uint32_t* pixel_index,
									size_t capacity, size_t* n_out);

/* -- unit-level material calls: IMaterial::eval / ::sample (src/core/material/IMaterial.h:15-55) */
prb_status prb_material_eval(prb_ctx* ctx, const prb_material_query* q, size_t n, prb_material_result* out);
prb_status prb_material_sample(prb_ctx* ctx, const prb_material_query* q, size_t n, prb_material_result* out);

prb_status prb_get_stats(prb_ctx* ctx, prb_stats* out);
prb_status prb_reset_stats(prb_ctx* ctx);
/* device time (ms, CUDA events on the context stream) spent in the last prb_render_tiles / prb_trace_* call */
prb_status prb_last_device_ms(prb_ctx* ctx, float* ms);


/* -- per-stage device times of the wavefront kernels (the analogue of the reference's PR_PROFILE scope timers,
 * src/base/Profiler.h:53-106).  While enabled, prb_render_tiles launches the stage kernels directly (no CUDA-graph
 * replay) with a CUDA-event pair around every launch on the context stream and accumulates ms[] / launches[] per stage:
 * PRB_STAGE_TRACE (k_trace: shadow any-hit + closest hit), PRB_STAGE_SHADE (k_shade: shading, NEE, scattering, film,
 * camera-sample regeneration).  Arrays hold PRB_STAGE__COUNT entries. */
enum { PRB_STAGE_TRACE = 0, PRB_STAGE_SHADE = 1, PRB_STAGE__COUNT = 2 };
prb_status prb_set_profiling(prb_ctx* ctx, int enabled);
prb_status prb_get_stage_times(prb_ctx* ctx, float* ms, uint64_t* launches);

/* -- shading path.  The shading stage exists in two bit-identical forms: ONE kernel (k_shade, slots sorted by material per
 * block) or STAGED (k_shade_geom, then k_shade_nee / k_shade_scatter once per material type over compact queues).  Which is
 * faster depends on the scene, so by default (PRB_SHADING_AUTO) a context times both during the first poll intervals of the
 * first render after prb_upload_scene and keeps the faster one.  prb_set_shading_mode pins it (also: environment variable
 * PRB_STAGED=0|1); prb_get_shading_mode reports the current choice, PRB_SHADING_AUTO while still undecided. */
enum { PRB_SHADING_AUTO = -1, PRB_SHADING_SINGLE = 0, PRB_SHADING_STAGED = 1 };
prb_status prb_set_shading_mode(prb_ctx* ctx, int mode);
prb_status prb_get_shading_mode(prb_ctx* ctx, int* mode);

/* -- the integrator prb_render_tiles runs.  PRB_INTEGRATOR_DIRECT: the path tracer above (reference direct.cpp).
 * PRB_INTEGRATOR_AO: ambient occlusion (reference plugins/main/integrators/ao.cpp): per sample the camera ray of 'direct' (same
 * draws) and its closest hit; a miss adds a zero sample and counts no sample; a hit writes the first-hit AOVs and sample count
 * like 'direct' and traces sample_count cosine-weighted rays about the (unflipped) shading normal any-hit from the safe-position
 * origin (tmin 1e-4, counted as shadow rays); the sample's value is 1 - occluded / sample_count, pushed as one fragment with the
 * MIS weight of a zero-radiance miss (heroFactor / (WavelengthPDF * sum heroFactor)) and importance 1.  Films, tiles, resume,
 * reductions, stats and timings mean the same as under 'direct'; with profiling on, the primary and occlusion kernels count as
 * PRB_STAGE_TRACE and the film fold as PRB_STAGE_SHADE.
 * PRB_INTEGRATOR_VF: visual feedback, the debug view of scene set-up (reference plugins/main/integrators/visualfeedback.cpp):
 * per sample the camera ray of 'direct' (same draws) and its closest hit.  A miss is handled as under 'ao'.  A hit writes the
 * first-hit AOVs and sample count like 'direct' and one linear-sRGB colour c chosen by `mode` (PRB_VF_*):
 *   ENTITY_ID palette(entity id)           MATERIAL_ID palette(material id), black for PRB_INVALID_ID
 *   EMISSION_ID palette(emission id), black for PRB_INVALID_ID    PRIMITIVE_ID palette(face index; 0 for spheres and planes)
 *   PARAMETER (u, v, 0) of the first-hit AOV   INSIDE (1, 0, 0) when dot(D, N) > 0 (back face), else (0, 1, 0)
 *   NDOTV |dot(N, D)| (1, 1, 1)            (D: the normalised camera direction, N: the geometry normal of the hit)
 * palette(id), in fp32: h = frac(id * 0.618034), S = 0.7, V = 0.9, then the textbook HSV -> RGB.  The sample's value is
 * XYZ = M c with M the sRGB (D65) RGB -> XYZ matrix, folded into the film as it is, without the spectral fragment path (also
 * on a monotonic film), so the sRGB tone mode of the film gives back c.  The RNG stream ends after the camera draws.  Films,
 * tiles, resume, reductions, stats and timings mean the same as under 'ao'; with profiling on, its one kernel counts as
 * PRB_STAGE_TRACE.
 * prb_upload_scene resets the integrator to { PRB_INTEGRATOR_DIRECT, 0 }.  prb_set_integrator fails with PRB_ERR_NO_SCENE before
 * a scene was uploaded, PRB_ERR_INVALID_ARG for an unknown type, 'ao' with sample_count 0 or 'vf' with an unknown mode,
 * PRB_ERR_UNSUPPORTED for 'ao' or 'vf' on a scene with light path expression channels. */
enum { PRB_INTEGRATOR_DIRECT = 0, PRB_INTEGRATOR_AO = 1, PRB_INTEGRATOR_VF = 2 };
enum { PRB_VF_ENTITY_ID, PRB_VF_MATERIAL_ID, PRB_VF_EMISSION_ID, PRB_VF_PRIMITIVE_ID, PRB_VF_PARAMETER, PRB_VF_INSIDE, PRB_VF_NDOTV, PRB_VF__COUNT };
/* 8 bytes: the parameter of each integrator shares the second word, so records of existing callers keep their size */
typedef struct prb_integrator {
	uint32_t type; /* PRB_INTEGRATOR_* */
	union {
		uint32_t sample_count; /* AO: occlusion rays per pixel sample (reference parameter 'sample_count', default 10) */
		uint32_t mode;		   /* VF: PRB_VF_* (reference parameter 'mode', default colored_entity_id) */
	};
} prb_integrator;
prb_status prb_set_integrator(prb_ctx* ctx, const prb_integrator* integrator);
prb_status prb_get_integrator(prb_ctx* ctx, prb_integrator* out);

#ifdef __cplusplus
}
#endif
#endif /* PRB200_ABI_H */
