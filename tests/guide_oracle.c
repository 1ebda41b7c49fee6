/* tests/guide_oracle.c — TEST INFRASTRUCTURE: the CPU oracle of all five AOV planes (McAovTargets, include/mcskin_cuda.h),
 * guide planes (normal, albedo) included.  The frame walk is tests/aov_oracle.c's; this unit adds the guides' fold.
 *
 * It compiles the unmodified CPU oracle (oracle/mcskin_oracle.c) into the same unit and walks a frame exactly as that
 * oracle's render_tile does (tile_renderer.cpp:71-127): the tiles of generateTiles, each with its own stream seeded
 * tile.y * width + tile.x (either rng_mode); per pixel, per sample in order, the jitter draws (spp > 1), (u, v), the
 * pinhole or thin-lens ray with its lens draws; and the re-test intersectScene of that ray (tile_renderer.cpp:111, the
 * query whose miss gives the sample the gradient).  The planes fold those hits in sample order:
 *   coverage = (float)n * (1.0f / (float)spp), depth = left-to-right sum of t over the hits / (float)n (0 if n == 0),
 *   tri_id = box*12 + face*2 of the first hit (-1 if n == 0);
 *   normal, albedo (when given) = left-to-right sums of h.normal and h.tex_color over the hits, each component / (float)n
 *   (zeros if n == 0).
 * Shading draws nothing from a tile's stream, so the colour path (mcorc_render) is not needed to reproduce the rays.
 * Built with the oracle's own flags (oracle/Makefile): no FMA contraction, no fast-math. */
#include "../oracle/mcskin_oracle.c"

int32_t guideorc_render_aovs(const McScene* sc, const McConfig* cfg, const McAovTargets* aov) {
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
    for (int t = 0; t < nTiles; ++t) {
        const McTile* tile = &tiles[t];
        Mt rng;
        mt_seed_mode(&rng, (uint32_t)(tile->y * cfg->width + tile->x), cfg->rng_mode == MC_RNG_COUNTER);
        for (int py = tile->y; py < tile->y + tile->height; ++py)
            for (int px = tile->x; px < tile->x + tile->width; ++px) {
                int n = 0, firstId = -1;
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
                        if (n == 0) firstId = h.box * 12 + h.face * 2;
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
            }
    }
    free(tiles);
    return 0;
}
