/* tests/texel_oracle.c — TEST INFRASTRUCTURE: the CPU oracle of all six AOV planes (McAovTargets, include/mcskin_cuda.h),
 * the texel plane included.  The frame walk is tests/guide_oracle.c's (itself tests/aov_oracle.c's); this unit adds the
 * texel plane's fold.
 *
 * It compiles the unmodified CPU oracle (oracle/mcskin_oracle.c) into the same unit and walks a frame exactly as that
 * oracle's render_tile does: the tiles of generateTiles, each with its own stream seeded tile.y * width + tile.x (either
 * rng_mode); per pixel, per sample in order, the jitter draws (spp > 1), (u, v), the pinhole or thin-lens ray with its
 * lens draws; and the re-test intersect_scene of that ray.  The planes fold those hits in sample order:
 *   coverage, depth, tri_id, normal, albedo as tests/guide_oracle.c folds them;
 *   texel = the texel index of the first hit (-1 if n == 0).
 *
 * McHit carries no texel index, so the index is restated for the winning box only: the local ray of a posed box (as
 * intersect_mesh builds it), the slab walk, entry or exit face (as intersect_box picks them), face_uv, and
 * sample_face's addressing; for an outer layer whose first face texel has alpha 0, the exit face's texel.  A face
 * without texels gives the synthetic texels past the pool: n_texels (null texture) and n_texels + 1 (empty region).
 * Every hit checks the restatement against the oracle itself: the texel's RGBA (or the synthetic colour) must equal
 * McHit.tex_color bit for bit and the face must equal McHit.face; otherwise the call fails with -2 and says where.
 * Built with the oracle's own flags (oracle/Makefile): no FMA contraction, no fast-math. */
#include <stdio.h>

#include "../oracle/mcskin_oracle.c"

/* sample_face's addressing (texture_region.h:19-26) as a pool index, with the two synthetic texels past the pool */
static int texel_index(const McScene* sc, const McFaceTex* ft, float u, float v) {
    if (ft->texel_offset < 0) return sc->n_texels;
    if (ft->width <= 0 || ft->height <= 0) return sc->n_texels + 1;
    int x = (int)(u * ft->width);
    int y = (int)(v * ft->height);
    x = x < 0 ? 0 : (x > ft->width - 1 ? ft->width - 1 : x);
    y = y < 0 ? 0 : (y > ft->height - 1 ? ft->height - 1 : y);
    return ft->texel_offset + y * ft->width + x;
}
static Col texel_color(const McScene* sc, int texel) {
    if (texel == sc->n_texels) return col(1, 0, 1, 1);
    if (texel == sc->n_texels + 1) return col(0, 0, 0, 1);
    const float* p = sc->texels_rgba + 4 * (size_t)texel;
    return col(p[0], p[1], p[2], p[3]);
}

/* The texel and face intersect_mesh's hit on box b took, for a ray known to hit that box. */
static int hit_texel_of(const McScene* sc, V3 ro, V3 rd, int b, int* faceOut) {
    const McBox* box = &sc->boxes[b];
    if (box->has_rotation) {  /* intersect_mesh: the ray in the box's own frame */
        V3 pivot = v3(box->pivot[0], box->pivot[1], box->pivot[2]);
        V3 lo = rotate_point(ro, pivot, 0, -box->rot_z_deg);
        lo = rotate_point(lo, pivot, -box->rot_x_deg, 0);
        V3 ld = rotate_dir(rd, 0, -box->rot_z_deg);
        ld = rotate_dir(ld, -box->rot_x_deg, 0);
        ro = lo;
        rd = vnorm(ld);
    }
    const float* lo = box->bounds_min;
    const float* hi = box->bounds_max;
    const float o[3] = {ro.x, ro.y, ro.z}, d[3] = {rd.x, rd.y, rd.z};
    /* intersect_box's slab walk; the box is hit, so none of its early returns is taken */
    float tmin = -FLT_MAX, tmax = FLT_MAX;
    int axis = 0, neg = 0;
    for (int i = 0; i < 3; ++i) {
        if (fabsf(d[i]) < 1e-8f) continue;
        float inv = 1.0f / d[i];
        float t0 = (lo[i] - o[i]) * inv, t1 = (hi[i] - o[i]) * inv;
        int en = 1;
        if (t0 > t1) { float t = t0; t0 = t1; t1 = t; en = 0; }
        if (t0 > tmin) { tmin = t0; axis = i; neg = en; }
        tmax = (t1 < tmax) ? t1 : tmax;
    }
    float tHit = tmin;
    if (tHit < 0.0f) {  /* origin inside: the exit face */
        tHit = tmax;
        exit_face(o, d, lo, hi, &axis, &neg);
    }
    V3 n;
    int f = face_of(axis, neg, &n);
    float u, v;
    face_uv(vadd(ro, vmul(rd, tHit)), lo, hi, axis, neg, &u, &v);
    int texel = texel_index(sc, &box->face[f], u, v);
    if (texel_color(sc, texel).a == 0.0f) {  /* an outer layer's alpha-0 texel: the exit face at tmax */
        int ea, en;
        exit_face(o, d, lo, hi, &ea, &en);
        f = face_of(ea, en, &n);
        face_uv(vadd(ro, vmul(rd, tmax)), lo, hi, ea, en, &u, &v);
        texel = texel_index(sc, &box->face[f], u, v);
    }
    *faceOut = f;
    return texel;
}

int32_t texelorc_render_aovs(const McScene* sc, const McConfig* cfg, const McAovTargets* aov) {
    if (!sc || !cfg || !aov) return -1;
    const size_t pixels = cfg->width > 0 && cfg->height > 0 ? (size_t)cfg->width * (size_t)cfg->height : 0;
    for (size_t i = 0; i < pixels; ++i) {
        if (aov->coverage) aov->coverage[i] = 0.0f;
        if (aov->depth) aov->depth[i] = 0.0f;
        if (aov->tri_id) aov->tri_id[i] = -1;
        for (int k = 0; k < 3; ++k)
            if (aov->normal) aov->normal[3 * i + k] = 0.0f;
        for (int k = 0; k < 4; ++k)
            if (aov->albedo) aov->albedo[4 * i + k] = 0.0f;
        if (aov->texel) aov->texel[i] = -1;
    }
    const int nTiles = mcorc_generate_tiles(cfg->width, cfg->height, cfg->tile_size, NULL, 0);
    if (nTiles == 0) return 0;
    McTile* tiles = (McTile*)malloc(sizeof(McTile) * (size_t)nTiles);
    mcorc_generate_tiles(cfg->width, cfg->height, cfg->tile_size, tiles, nTiles);
    Ctx cx;
    memset(&cx, 0, sizeof(cx));
    cx.sc = sc;
    cx.cfg = cfg;
    const float aspect = (float)cfg->width / (float)cfg->height;
    const int spp = cfg->samples_per_pixel > 1 ? cfg->samples_per_pixel : 1;
    float focusDist = cfg->focus_distance;
    if (focusDist <= 0.0f) {
        V3 pos = v3(sc->cam_pos[0], sc->cam_pos[1], sc->cam_pos[2]);
        V3 tgt = v3(sc->cam_target[0], sc->cam_target[1], sc->cam_target[2]);
        focusDist = vlen(vsub(tgt, pos));
    }
    int32_t rc = 0;
    for (int t = 0; t < nTiles && rc == 0; ++t) {
        const McTile* tile = &tiles[t];
        Mt rng;
        mt_seed_mode(&rng, (uint32_t)(tile->y * cfg->width + tile->x), cfg->rng_mode == MC_RNG_COUNTER);
        for (int py = tile->y; py < tile->y + tile->height; ++py)
            for (int px = tile->x; px < tile->x + tile->width; ++px) {
                int n = 0, firstId = -1, firstTexel = -1;
                float tSum = 0.0f, nSum[3] = {0.0f, 0.0f, 0.0f}, cSum[4] = {0.0f, 0.0f, 0.0f, 0.0f};
                for (int s = 0; s < spp; ++s) {
                    float jx = (spp == 1) ? 0.5f : canonical_float(&rng);
                    float jy = (spp == 1) ? 0.5f : canonical_float(&rng);
                    float u = ((float)px + jx) / (float)cfg->width;
                    float v = ((float)py + jy) / (float)cfg->height;
                    V3 ro, rd;
                    if (cfg->dof_enabled && cfg->aperture > 1e-6f) dof_ray(sc, u, v, aspect, cfg->aperture, focusDist, &rng, &ro, &rd);
                    else camera_ray(sc, u, v, aspect, &ro, &rd);
                    McHit h = intersect_scene(&cx, ro, rd);
                    if (h.hit) {
                        int face;
                        const int texel = hit_texel_of(sc, ro, rd, h.box, &face);
                        const Col c = texel_color(sc, texel);
                        const float rgba[4] = {c.r, c.g, c.b, c.a};
                        if (face != h.face || memcmp(rgba, h.tex_color, sizeof(rgba)) != 0) {
                            fprintf(stderr, "texel oracle: pixel (%d, %d) sample %d, box %d: restated face %d texel %d, "
                                    "oracle face %d\n", px, py, s, h.box, face, texel, h.face);
                            rc = -2;
                        }
                        if (n == 0) {
                            firstId = h.box * 12 + h.face * 2;
                            firstTexel = texel;
                        }
                        ++n;
                        tSum += h.t;
                        for (int k = 0; k < 3; ++k) nSum[k] += h.normal[k];
                        for (int k = 0; k < 4; ++k) cSum[k] += h.tex_color[k];
                    }
                }
                const size_t i = (size_t)py * cfg->width + px;
                const float inv = 1.0f / (float)spp;
                if (aov->coverage) aov->coverage[i] = (float)n * inv;
                if (aov->depth) aov->depth[i] = n > 0 ? tSum / (float)n : 0.0f;
                if (aov->tri_id) aov->tri_id[i] = firstId;
                for (int k = 0; k < 3; ++k)
                    if (aov->normal) aov->normal[3 * i + k] = n > 0 ? nSum[k] / (float)n : 0.0f;
                for (int k = 0; k < 4; ++k)
                    if (aov->albedo) aov->albedo[4 * i + k] = n > 0 ? cSum[k] / (float)n : 0.0f;
                if (aov->texel) aov->texel[i] = firstTexel;
            }
    }
    free(tiles);
    return rc;
}
