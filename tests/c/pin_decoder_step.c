/*
 * pin_decoder_step.c -- pins oracle/vox_oracle.c:orc_decoder_layer_step (+ final norm, logits, argmax) against the UNMODIFIED
 * reference's vox_decoder_forward (voxtral_decoder.c:586-706) at the model's real dimensions.
 *
 * The reference's structs are public (voxtral.h:100-204), so a vox_ctx_t can be filled by hand: every layer points at the same
 * seven random bf16 matrices (233 MB instead of 6 GB) but has its own norm weights and ada_scale row, so a layer-indexing slip
 * would still show.  Three consecutive forwards exercise the KV cache (positions 0, 1, 2).
 * Built and run by tests/test_cpu_oracle.py: writes the restatement's logits of step s to <dir>/orc_<s>.f32.  Built with
 * -DPIN_REFERENCE and linked with the reference, it also writes the reference's logits to <dir>/ref_<s>.f32 and its greedy id
 * and KV length to <dir>/ref_<s>.i32: what the test records (include/voxtral_b200.h declares the same structs and functions).
 */
#include "voxtral_b200.h"
#include "vox_oracle.h"

#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static uint32_t g_rng = 0xB2000001u;
static float urand(void) { g_rng = g_rng * 1664525u + 1013904223u; return (float)(g_rng >> 8) * (1.0f / 16777216.0f); }
static uint16_t f2bf(float f) { uint32_t u; memcpy(&u, &f, 4); return (uint16_t)((u + 0x7fffu + ((u >> 16) & 1u)) >> 16); }
static uint16_t *rand_bf16(size_t rows, size_t cols, float scale) {
    uint16_t *w = malloc(rows * cols * 2);
    for (size_t i = 0; i < rows * cols; i++) w[i] = f2bf((urand() * 2.0f - 1.0f) * scale);
    return w;
}
static float *rand_f32(size_t n, float centre, float spread) {
    float *w = malloc(n * 4);
    for (size_t i = 0; i < n; i++) w[i] = centre + (urand() * 2.0f - 1.0f) * spread;
    return w;
}
static int write_file(const char *dir, const char *name, int s, const char *ext, const void *p, size_t bytes) {
    char path[4096];
    snprintf(path, sizeof path, "%s/%s_%d.%s", dir, name, s, ext);
    FILE *f = fopen(path, "wb");
    if (!f || fwrite(p, 1, bytes, f) != bytes) return 1;
    return fclose(f) != 0;
}

int main(int argc, char **argv) {
    if (argc != 2) return 2;
    const int D = VOX_DEC_DIM, H = VOX_DEC_HIDDEN, QD = VOX_DEC_HEADS * VOX_DEC_HEAD_DIM, KVD = VOX_DEC_KV_HEADS * VOX_DEC_HEAD_DIM;
    vox_ctx_t *ctx = calloc(1, sizeof *ctx);
    ctx->use_bf16 = 1;
    ctx->delay_tokens = 6;
    uint16_t *wq = rand_bf16(QD, D, sqrtf(3.0f / D)), *wk = rand_bf16(KVD, D, sqrtf(3.0f / D)), *wv = rand_bf16(KVD, D, sqrtf(3.0f / D));
    uint16_t *wo = rand_bf16(D, QD, 0.3f * sqrtf(3.0f / QD));
    uint16_t *w1 = rand_bf16(H, D, sqrtf(3.0f / D)), *w3 = rand_bf16(H, D, sqrtf(3.0f / D)), *w2 = rand_bf16(D, H, 0.3f * sqrtf(3.0f / H));
    ctx->decoder.tok_embeddings_bf16 = rand_bf16(VOX_VOCAB_SIZE, D, 0.05f);
    ctx->decoder.norm = rand_f32(D, 1.0f, 0.2f);
    ctx->ada_scale = rand_f32((size_t)VOX_DEC_LAYERS * D, 0.0f, 0.1f);
    orc_dec_layer L[VOX_DEC_LAYERS];
    for (int l = 0; l < VOX_DEC_LAYERS; l++) {
        vox_dec_layer_t *y = &ctx->decoder.layers[l];
        y->wq_weight_bf16 = wq; y->wk_weight_bf16 = wk; y->wv_weight_bf16 = wv; y->wo_weight_bf16 = wo;
        y->w1_weight_bf16 = w1; y->w2_weight_bf16 = w2; y->w3_weight_bf16 = w3;
        y->attention_norm = rand_f32(D, 1.0f, 0.3f); y->ffn_norm = rand_f32(D, 1.0f, 0.3f);
        L[l].wq = wq; L[l].wk = wk; L[l].wv = wv; L[l].wo = wo; L[l].w1 = w1; L[l].w2 = w2; L[l].w3 = w3;
        L[l].attn_norm = y->attention_norm; L[l].ffn_norm = y->ffn_norm; L[l].ada_scale = ctx->ada_scale + (size_t)l * D;
    }
#ifdef PIN_REFERENCE
    /* kv_cache_grow() doubles kv_cache_max and never terminates from 0; the stream path always allocates first */
    if (vox_decoder_kv_cache_preallocate(ctx, 16) != 0) return 3;
#endif
    const int steps = 3, max_seq = 8;
    float *kc = calloc((size_t)VOX_DEC_LAYERS * max_seq * KVD, 4), *vc = calloc((size_t)VOX_DEC_LAYERS * max_seq * KVD, 4);
    float *logits_orc = malloc((size_t)VOX_VOCAB_SIZE * 4);
    float *x = malloc(D * 4), *xn = malloc(D * 4), *emb = malloc(D * 4);
    int bad = 0;
    for (int s = 0; s < steps; s++) {
        for (int i = 0; i < D; i++) emb[i] = (urand() * 2.0f - 1.0f) * 1.5f;
#ifdef PIN_REFERENCE
        float *logits_ref = malloc((size_t)VOX_VOCAB_SIZE * 4);
        int ref_ids[2] = { vox_decoder_forward(ctx, emb, logits_ref), 0 };
        ref_ids[1] = ctx->kv_cache_len;
        bad |= write_file(argv[1], "ref", s, "f32", logits_ref, (size_t)VOX_VOCAB_SIZE * 4);
        bad |= write_file(argv[1], "ref", s, "i32", ref_ids, sizeof ref_ids);
        free(logits_ref);
#endif
        memcpy(x, emb, D * 4);
        for (int l = 0; l < VOX_DEC_LAYERS; l++)
            orc_decoder_layer_step(x, &L[l], kc + (size_t)l * max_seq * KVD, vc + (size_t)l * max_seq * KVD, s, s, D, VOX_DEC_HEADS,
                                   VOX_DEC_KV_HEADS, VOX_DEC_HEAD_DIM, H, VOX_DEC_WINDOW, VOX_ROPE_THETA, VOX_DEC_NORM_EPS);
        orc_rms_norm(xn, x, ctx->decoder.norm, 1, D, VOX_DEC_NORM_EPS);
        orc_linear_bf16(logits_orc, xn, ctx->decoder.tok_embeddings_bf16, NULL, 1, D, VOX_VOCAB_SIZE);
        bad |= write_file(argv[1], "orc", s, "f32", logits_orc, (size_t)VOX_VOCAB_SIZE * 4);
    }
    return bad;
}
