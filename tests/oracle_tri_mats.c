/*
 * tests/oracle_tri_mats.c — the CPU oracle (oracle/ipt_oracle.c) with per-triangle materials, the checker of
 * ipt_scene_set_triangle_materials. TEST INFRASTRUCTURE ONLY, built by tests/oracle_tri_mats.py.
 *
 * The oracle is compiled here unchanged, with one hook: its trace_geometry reports `d->triangle_material` for a hit on
 * triangle `best - d->n_prims`, the only place that reads the field. The macro below turns that read into
 * `d->triangle_material + delta`, where delta (mod 2^32) makes the sum the index attached to that triangle, or 0 where
 * nothing is attached. A macro is not expanded inside its own expansion, so the field keeps its name. Everything the
 * oracle computes from that hit (render, mix sample, mix value) then sees the attached material; without an attachment it
 * is the oracle bit for bit (tests/test_oracle_mesh_materials.py checks both).
 */
#define _GNU_SOURCE
#include "ipt_b200.h"

#include <stdint.h>
#include <stdlib.h>
#include <string.h>

/* Per-triangle materials attached to a description, in a small table keyed by the description's address. Each entry
 * holds a copy of the caller's n_triangles indices. */
#define TRI_MATS_SLOTS 64
static struct { const ipt_scene_desc* d; uint32_t* mats; } g_tri_mats[TRI_MATS_SLOTS];

static uint32_t tri_mat_delta(const ipt_scene_desc* d, uint32_t best) {
    for (int i = 0; i < TRI_MATS_SLOTS; ++i)
        if (g_tri_mats[i].d == d) return g_tri_mats[i].mats[best - d->n_prims] - d->triangle_material;
    return 0;
}

/* Attach materials[k] (an index into d->materials) to triangle k of d; NULL detaches. Returns 0, 1 if an index is out of
 * range, 2 if the table is full. */
int ipt_oracle_set_triangle_materials(const ipt_scene_desc* d, const uint32_t* materials) {
    int slot = -1;
    for (int i = 0; i < TRI_MATS_SLOTS; ++i)
        if (g_tri_mats[i].d == d) slot = i;
    if (!materials) {
        if (slot >= 0) { free(g_tri_mats[slot].mats); g_tri_mats[slot].d = NULL; g_tri_mats[slot].mats = NULL; }
        return 0;
    }
    for (uint64_t k = 0; k < d->n_triangles; ++k)
        if (materials[k] >= d->n_materials) return 1;
    for (int i = 0; slot < 0 && i < TRI_MATS_SLOTS; ++i)
        if (!g_tri_mats[i].d) slot = i;
    if (slot < 0) return 2;
    uint32_t* copy = (uint32_t*)malloc(sizeof(uint32_t) * (d->n_triangles ? d->n_triangles : 1));
    memcpy(copy, materials, sizeof(uint32_t) * d->n_triangles);
    free(g_tri_mats[slot].mats);
    g_tri_mats[slot].d = d;
    g_tri_mats[slot].mats = copy;
    return 0;
}

#define triangle_material triangle_material + tri_mat_delta(d, best)
#include "ipt_oracle.c"
#undef triangle_material
