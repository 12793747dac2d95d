/* The 13 OpenImageDenoise C entry points Utils::OIDN_denoise uses (source/utils.cpp:144-196), implemented over the library's own
 * GPU denoise stage (b200rt_denoise_guided, csrc/denoise.cu). The reference does not ship the OIDN binaries; with this file its
 * unmodified main.cpp links, runs end to end, and the three "denoised" PNGs it writes (main.cpp:118-125) are filtered on the GPU.
 * Not OIDN: an edge-avoiding a-trous filter in OIDN's place (DESIGN.md). Implemented: the float3 "color" image filtered into
 * "output" (the reference binds both names to the same buffer, utils.cpp:158-159), and the RT filter's optional float3 auxiliary
 * images "albedo" and "normal", which become the filter's edge-stopping guides (b200rt_render_aovs computes them). The reference sets
 * neither, so its PNGs are filtered by colour alone. Bool parameters ("hdr", "cleanAux", ...) are accepted and ignored. Images in
 * another format, at a byte offset or with other strides are refused (oidnGetDeviceError reports it). */
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "b200rt.h"

typedef struct { void* data; size_t bytes; } nbuf;
typedef struct { nbuf* color; nbuf* output; nbuf* albedo; nbuf* normal; size_t w, h; const char* bad; } nfilter;
static int g_dev;
static const char* g_err;

void* oidnNewDevice(int type) { (void)type; return &g_dev; }
void oidnCommitDevice(void* d) { (void)d; }
void* oidnNewBuffer(void* d, size_t bytes) { (void)d; nbuf* b = (nbuf*)malloc(sizeof(nbuf)); b->data = malloc(bytes); b->bytes = bytes; return b; }
void* oidnGetBufferData(void* b) { return ((nbuf*)b)->data; }
void* oidnNewFilter(void* d, const char* type) { (void)d; (void)type; return calloc(1, sizeof(nfilter)); }
/* Only packed float3 images are understood: anything else is refused with a device error (and the filter will not run) instead of
 * being read as packed float3. OIDN's strides of 0 mean "packed"; the explicit packed strides are accepted too. */
void oidnSetFilterImage(void* f, const char* name, void* buf, int fmt, size_t w, size_t h, size_t off, size_t ps, size_t rs)
{
    nfilter* flt = (nfilter*)f;
    const char* bad = fmt != 3 ? "image format not supported (only OIDN_FORMAT_FLOAT3)"
                    : off != 0 ? "image byte offset not supported (must be 0)"
                    : ps != 0 && ps != 12 ? "image pixel stride not supported (must be 0 or 12)"
                    : rs != 0 && rs != 12 * w ? "image row stride not supported (must be 0 or 12 * width)" : NULL;
    if (bad) { g_err = flt->bad = bad; return; }
    if (!strcmp(name, "color")) flt->color = (nbuf*)buf;
    else if (!strcmp(name, "output")) flt->output = (nbuf*)buf;
    else if (!strcmp(name, "albedo")) flt->albedo = (nbuf*)buf;
    else if (!strcmp(name, "normal")) flt->normal = (nbuf*)buf;
    flt->w = w; flt->h = h;
}
void oidnSetFilterBool(void* f, const char* name, int v) { (void)f; (void)name; (void)v; }
void oidnCommitFilter(void* f) { (void)f; }
void oidnExecuteFilter(void* f)
{
    nfilter* flt = (nfilter*)f;
    if (flt->bad) { g_err = flt->bad; return; }
    if (!flt->color || !flt->output) { g_err = "color / output image not set"; return; }
    if (b200rt_denoise_guided((const float*)flt->color->data, 3, flt->albedo ? (const float*)flt->albedo->data : NULL,
                              flt->normal ? (const float*)flt->normal->data : NULL, (int)flt->w, (int)flt->h, 1.0f, 0, 0.0f,
                              (float*)flt->output->data))
        g_err = b200rt_last_error();
}
int oidnGetDeviceError(void* d, const char** msg) { (void)d; if (msg) *msg = g_err; const int e = g_err != 0; g_err = 0; return e; }
void oidnReleaseBuffer(void* b) { if (b) { free(((nbuf*)b)->data); free(b); } }
void oidnReleaseFilter(void* f) { free(f); }
void oidnReleaseDevice(void* d) { (void)d; }
