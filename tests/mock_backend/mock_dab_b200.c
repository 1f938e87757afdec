/*
 * mock_dab_b200.c — TEST DOUBLE of the C ABI (include/dab_b200.h) for exercising the host glue on a machine without a GPU.
 *
 * NOT part of the product and never built into the tree: tests/test_glue_mock.py compiles it into a temporary directory as
 * "libdab_b200.so" and runs welle.io_b200/glue_test and welle.io_b200/batch_decode with LD_LIBRARY_PATH pointing there.  It does no
 * signal processing of its own: at dabb_create it loads the IQ files named by $DABB_MOCK_IQ (':'-separated, one per stream) and lets
 * the oracle (oracle/liboracle.so, test infrastructure) decode each whole stream; dabb_process() then hands out one frame record per
 * stream after the other (FIBs, CRC mask, correctors, logical frames) in the layout of the ABI.  RS statistics, superframes and the diagnostic taps are not served (the GPU tests cover them).
 * Only the entry points the glue calls are implemented.
 */
#include "../../include/dab_b200.h"
#include "../../oracle/dab_oracle.h"

#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

typedef struct {
    float* iq; long n;
    long frames; uint8_t* fibs; orc_frame_info_t* info;
    int k;                                   /* next frame to hand out */
    int sel_frame; int sel_slot; int flen; uint8_t* msc; long n_msc;
} mock_stream;
struct dabb_ctx {
    int S; mock_stream* st;
    int disable_coarse, placement, freqsync;
    char err[128];
};

static long run_oracle(mock_stream* c, const orc_rx_cfg_t* cfg, uint8_t* fibs, long fib_cap, uint8_t* msc, long msc_cap, long* n_msc, orc_frame_info_t* info, long info_cap)
{
    orc_rx_t* rx = orc_rx_new(cfg);
    long nf = 0, nm = 0, nr = 0;
    int* rs = (int*)malloc(sizeof(int) * 2 * 4 * (size_t)info_cap);
    const long frames = orc_rx_run(rx, c->iq, c->n, fibs, fib_cap, &nf, msc, msc_cap, &nm, rs, 4 * info_cap, &nr, info, info_cap, NULL, 0);
    free(rs); orc_rx_free(rx);
    if (n_msc) *n_msc = nm;
    return frames;
}

int dabb_abi_version(void) { return DABB_ABI_VERSION; }
const char* dabb_last_error(const dabb_ctx* c) { return c ? c->err : "mock backend"; }

int dabb_create(const dabb_config* cfg, dabb_ctx** out)
{
    if (!cfg || !out || cfg->abi_version != DABB_ABI_VERSION || cfg->n_streams < 1) return DABB_E_ARG;
    const char* list = getenv("DABB_MOCK_IQ");               /* ':'-separated, one cf32 file per stream */
    if (!list) return DABB_E_NODEVICE;
    dabb_ctx* c = (dabb_ctx*)calloc(1, sizeof *c);
    c->S = cfg->n_streams; c->st = (mock_stream*)calloc((size_t)c->S, sizeof(mock_stream));
    c->disable_coarse = cfg->disable_coarse; c->placement = cfg->fft_placement; c->freqsync = cfg->freqsync_method;
    char* copy = strdup(list); char* save = NULL; char* tok = strtok_r(copy, ":", &save);
    for (int s = 0; s < c->S; s++, tok = strtok_r(NULL, ":", &save)) {
        mock_stream* z = &c->st[s];
        if (!tok) { free(copy); return DABB_E_ARG; }
        FILE* f = fopen(tok, "rb");
        if (!f) { free(copy); return DABB_E_ARG; }
        fseek(f, 0, SEEK_END); const long bytes = ftell(f); fseek(f, 0, SEEK_SET);
        z->n = bytes / 8; z->iq = (float*)malloc((size_t)bytes);
        if (fread(z->iq, 1, (size_t)bytes, f) != (size_t)bytes) { fclose(f); free(copy); return DABB_E_ARG; }
        fclose(f);
        const long cap = z->n / ORC_TF + 2;
        z->fibs = (uint8_t*)calloc((size_t)cap * 12, 33); z->info = (orc_frame_info_t*)calloc((size_t)cap, sizeof(orc_frame_info_t));
        orc_rx_cfg_t oc; memset(&oc, 0, sizeof oc);
        oc.disable_coarse = c->disable_coarse; oc.fft_placement = c->placement; oc.freqsync_method = c->freqsync;
        z->frames = run_oracle(z, &oc, z->fibs, cap * 12, NULL, 0, NULL, z->info, cap);
        z->sel_frame = -1;
    }
    free(copy);
    *out = c;
    return DABB_OK;
}
void dabb_destroy(dabb_ctx* c)
{
    if (!c) return;
    for (int s = 0; s < c->S; s++) { free(c->st[s].iq); free(c->st[s].fibs); free(c->st[s].info); free(c->st[s].msc); }
    free(c->st); free(c);
}
int dabb_stream_reset(dabb_ctx* c, int32_t first, int32_t count, int64_t pos) { (void)first; (void)count; (void)pos; return c ? DABB_OK : DABB_E_ARG; }
int dabb_set_options(dabb_ctx* c, const dabb_options* o) { return c && o ? DABB_OK : DABB_E_ARG; }

int dabb_select_subchannel(dabb_ctx* c, int32_t first, int32_t count, int32_t slot, const dabb_subchannel* sc)
{
    if (!c || !sc || slot < 0 || slot >= DABB_MAX_SUBCH || first < 0 || count < 1 || first + count > c->S) return DABB_E_ARG;
    for (int s = first; s < first + count; s++) {
        mock_stream* z = &c->st[s];
        orc_rx_cfg_t oc; memset(&oc, 0, sizeof oc);
        oc.disable_coarse = c->disable_coarse; oc.fft_placement = c->placement; oc.freqsync_method = c->freqsync;
        oc.subch_start_cu = sc->start_cu; oc.subch_len_cu = sc->length_cu; oc.dabplus = sc->dabplus; oc.select_after_frames = z->k;
        const int rc = sc->short_form ? orc_prot_uep(sc->bitrate, sc->uep_level, &oc.prot) : orc_prot_eep(sc->bitrate, sc->eep_profile_a, sc->eep_level, &oc.prot);
        if (rc) { snprintf(c->err, sizeof c->err, "unsupported protection"); return DABB_E_UNSUPPORTED; }
        const long cap = z->n / ORC_TF + 2;
        free(z->msc);
        z->flen = 3 * sc->bitrate;
        z->msc = (uint8_t*)calloc((size_t)cap * 4, (size_t)z->flen);
        uint8_t* fibs = (uint8_t*)calloc((size_t)cap * 12, 33); orc_frame_info_t* info = (orc_frame_info_t*)calloc((size_t)cap, sizeof *info);
        run_oracle(z, &oc, fibs, cap * 12, z->msc, cap * 4 * z->flen, &z->n_msc, info, cap);
        free(fibs); free(info);
        z->sel_frame = z->k; z->sel_slot = slot;
    }
    return DABB_OK;
}
int dabb_remove_subchannel(dabb_ctx* c, int32_t first, int32_t count, int32_t slot)
{
    (void)slot;
    if (!c || first < 0 || count < 1 || first + count > c->S) return DABB_E_ARG;
    for (int s = first; s < first + count; s++) c->st[s].sel_frame = -1;
    return DABB_OK;
}

int dabb_process(dabb_ctx* c, const dabb_io* io)
{
    if (!c || !io || !io->results) return DABB_E_ARG;
    /* a step of the real library takes time; at least 2 ms here too, so that what the glue does from other threads (the controller's
     * service selection) lands while its worker is decoding, however fast the host is */
    const struct timespec step = {0, 2000000};
    nanosleep(&step, NULL);
    for (int s = 0; s < c->S; s++) {
        mock_stream* z = &c->st[s];
        dabb_frame_result* r = &io->results[s];
        memset(r, 0, sizeof *r);
        if (io->buf_start && io->buf_start[s] < -(1LL << 30)) { r->status = DABB_FRAME_NEED_SAMPLES; continue; }    /* a window far behind the stream: parked */
        if (z->k >= z->frames) { r->status = DABB_FRAME_ACQUIRING; continue; }
        const orc_frame_info_t* fi = &z->info[z->k];
        r->status = DABB_FRAME_DECODED; r->start_index = fi->start_index; r->fine_corr = fi->fine; r->coarse_corr = fi->coarse; r->snr_raw = fi->snr_raw;
        r->next_pos = fi->frame_pos + ORC_TU + fi->start_index + 75L * ORC_TS + ORC_TNULL;
        for (int f = 0; f < 12; f++) {
            const uint8_t* rec = z->fibs + 33 * ((size_t)z->k * 12 + f);
            if (rec[0]) r->fib_crc_mask |= 1 << f;
            if (io->fibs) memcpy(io->fibs + ((size_t)s * 12 + f) * 32, rec + 1, 32);
        }
        /* the time de-interleaver delivers its first logical frame 16 CIFs (4 frames) after the selection took effect */
        if (z->sel_frame >= 0 && z->k >= z->sel_frame + 4 && io->msc) {
            const long first = ((long)(z->k - z->sel_frame - 4)) * 4;
            int n = 0;
            for (int q = 0; q < 4; q++) if ((first + q + 1) * z->flen <= z->n_msc) n++;
            r->n_logical[z->sel_slot] = n;
            uint8_t* dst = io->msc + (((size_t)s * DABB_MAX_SUBCH + (size_t)z->sel_slot) * 4) * (size_t)io->msc_stride;      /* [S][MAX_SUBCH][4][stride] */
            for (int q = 0; q < n; q++) memcpy(dst + (size_t)(4 - n + q) * io->msc_stride, z->msc + (size_t)(first + q) * z->flen, (size_t)z->flen);
        }
        z->k++;
    }
    return DABB_OK;
}
int dabb_read_tap(dabb_ctx* c, int32_t what, void* out, size_t bytes) { (void)c; (void)what; (void)out; (void)bytes; return DABB_E_STATE; }
