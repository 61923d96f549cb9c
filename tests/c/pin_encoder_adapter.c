/*
 * pin_encoder_adapter.c -- pins oracle/vox_oracle.c:orc_encoder_layer (x32 + final norm) and orc_adapter against the UNMODIFIED
 * reference's vox_encoder_forward_incremental (voxtral_encoder.c:452-636) and vox_adapter_forward (:642-674) at the model's real
 * dimensions, on a hand-filled public vox_ctx_t (all layers share seven random bf16 matrices, each has its own norms and biases).
 * vox_encoder_forward on 22 mel frames pins the conv stem (orc_conv_stem) + a cold-cache pass; two incremental calls (7 rows,
 * then 5) exercise the encoder K/V cache carry and the logical RoPE positions; both adapters run on the same 12 seeded rows.
 * Built and run by tests/test_cpu_oracle.py: writes the restatement's output of each check to <dir>/orc_<check>.f32.  Built with
 * -DPIN_REFERENCE and linked with the reference, it also writes the reference's to <dir>/ref_<check>.f32 and its encoder cache
 * length to <dir>/ref_enc_cache_len.i32: what the test records (include/voxtral_b200.h declares the same structs and functions).
 */
#include "voxtral_b200.h"
#include "vox_oracle.h"

#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

static uint32_t g_rng = 0xE2C0DE01u;
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
static int write_file(const char *dir, const char *side, const char *what, const char *ext, const void *p, size_t bytes) {
    char path[4096];
    snprintf(path, sizeof path, "%s/%s_%s.%s", dir, side, what, ext);
    FILE *f = fopen(path, "wb");
    if (!f || fwrite(p, 1, bytes, f) != bytes) return 1;
    return fclose(f) != 0;
}

int main(int argc, char **argv) {
    if (argc != 2) return 2;
    const int D = VOX_ENC_DIM, H = VOX_ENC_HIDDEN, QD = VOX_ENC_HEADS * VOX_ENC_HEAD_DIM;
    vox_ctx_t *ctx = calloc(1, sizeof *ctx);
    ctx->use_bf16 = 1;
    uint16_t *wq = rand_bf16(QD, D, sqrtf(3.0f / D)), *wk = rand_bf16(QD, D, sqrtf(3.0f / D)), *wv = rand_bf16(QD, D, sqrtf(3.0f / D));
    uint16_t *wo = rand_bf16(D, QD, 0.3f * sqrtf(3.0f / QD));
    uint16_t *w1 = rand_bf16(H, D, sqrtf(3.0f / D)), *w3 = rand_bf16(H, D, sqrtf(3.0f / D)), *w2 = rand_bf16(D, H, 0.3f * sqrtf(3.0f / H));
    orc_enc_layer L[VOX_ENC_LAYERS];
    for (int l = 0; l < VOX_ENC_LAYERS; l++) {
        vox_enc_layer_t *y = &ctx->encoder.layers[l];
        y->wq_weight_bf16 = wq; y->wk_weight_bf16 = wk; y->wv_weight_bf16 = wv; y->wo_weight_bf16 = wo;
        y->w1_weight_bf16 = w1; y->w2_weight_bf16 = w2; y->w3_weight_bf16 = w3;
        y->wq_bias = rand_f32(QD, 0.f, 0.05f); y->wv_bias = rand_f32(QD, 0.f, 0.05f);
        y->wo_bias = rand_f32(D, 0.f, 0.05f); y->w2_bias = rand_f32(D, 0.f, 0.05f);
        y->attention_norm = rand_f32(D, 1.0f, 0.3f); y->ffn_norm = rand_f32(D, 1.0f, 0.3f);
        L[l].wq = wq; L[l].wk = wk; L[l].wv = wv; L[l].wo = wo; L[l].w1 = w1; L[l].w2 = w2; L[l].w3 = w3;
        L[l].bq = y->wq_bias; L[l].bv = y->wv_bias; L[l].bo = y->wo_bias; L[l].b2 = y->w2_bias;
        L[l].attn_norm = y->attention_norm; L[l].ffn_norm = y->ffn_norm;
    }
    ctx->encoder.norm = rand_f32(D, 1.0f, 0.2f);
    ctx->adapter.linear0_weight_bf16 = rand_bf16(VOX_DEC_DIM, 4 * (size_t)D, sqrtf(3.0f / (4 * D)));
    ctx->adapter.linear1_weight_bf16 = rand_bf16(VOX_DEC_DIM, VOX_DEC_DIM, sqrtf(3.0f / VOX_DEC_DIM));

    ctx->encoder.conv0_weight = rand_f32((size_t)D * VOX_MEL_BINS * 3, 0.f, sqrtf(3.0f / (VOX_MEL_BINS * 3)));
    ctx->encoder.conv0_bias = rand_f32(D, 0.f, 0.05f);
    ctx->encoder.conv1_weight = rand_f32((size_t)D * D * 3, 0.f, sqrtf(3.0f / (D * 3)));
    ctx->encoder.conv1_bias = rand_f32(D, 0.f, 0.05f);

    int bad = 0;
    {   /* E4: whole-sequence encoder = conv stem + 32 layers from an empty cache + final norm */
        const int frames = 22, pos = 11;
        float *mel = rand_f32((size_t)frames * VOX_MEL_BINS, 0.2f, 0.8f);
#ifdef PIN_REFERENCE
        int n = 0;
        float *y_ref = vox_encoder_forward(ctx, mel, frames, &n);
        if (!y_ref || n != pos) return 5;
        bad |= write_file(argv[1], "ref", "encoder_full", "f32", y_ref, (size_t)pos * D * 4);
        free(y_ref);
#endif
        float *x = malloc((size_t)pos * D * 4);
        orc_conv_stem(x, mel, frames, ctx->encoder.conv0_weight, ctx->encoder.conv0_bias, ctx->encoder.conv1_weight, ctx->encoder.conv1_bias,
                      VOX_MEL_BINS, D);
        float *k1 = calloc((size_t)pos * QD, 4), *v1 = calloc((size_t)pos * QD, 4);
        for (int l = 0; l < VOX_ENC_LAYERS; l++)
            orc_encoder_layer(x, pos, &L[l], k1, v1, 0, 0, D, VOX_ENC_HEADS, VOX_ENC_HEAD_DIM, H, VOX_ENC_WINDOW, VOX_ROPE_THETA, VOX_ENC_NORM_EPS);
        orc_rms_norm(x, x, ctx->encoder.norm, pos, D, VOX_ENC_NORM_EPS);
        bad |= write_file(argv[1], "orc", "encoder_full", "f32", x, (size_t)pos * D * 4);
        free(x); free(k1); free(v1); free(mel);
    }

    const int calls[2] = { 7, 5 }, max_rows = 16;
    float *kc = calloc((size_t)VOX_ENC_LAYERS * max_rows * QD, 4), *vc = calloc((size_t)VOX_ENC_LAYERS * max_rows * QD, 4);
    int done = 0;
    for (int c = 0; c < 2; c++) {
        const int m = calls[c];
        float *xin = rand_f32((size_t)m * D, 0.f, 1.2f);
#ifdef PIN_REFERENCE
        int out_len = 0;
        float *y_ref = vox_encoder_forward_incremental(ctx, xin, m, &out_len);
        if (!y_ref || out_len != m) return 3;
        bad |= write_file(argv[1], "ref", c ? "encoder_call_2" : "encoder_call_1", "f32", y_ref, (size_t)m * D * 4);
        free(y_ref);
#endif
        float *x = malloc((size_t)m * D * 4);
        memcpy(x, xin, (size_t)m * D * 4);
        for (int l = 0; l < VOX_ENC_LAYERS; l++)
            orc_encoder_layer(x, m, &L[l], kc + (size_t)l * max_rows * QD, vc + (size_t)l * max_rows * QD, done, done, D, VOX_ENC_HEADS,
                              VOX_ENC_HEAD_DIM, H, VOX_ENC_WINDOW, VOX_ROPE_THETA, VOX_ENC_NORM_EPS);
        orc_rms_norm(x, x, ctx->encoder.norm, m, D, VOX_ENC_NORM_EPS);
        bad |= write_file(argv[1], "orc", c ? "encoder_call_2" : "encoder_call_1", "f32", x, (size_t)m * D * 4);
        done += m;
        free(x); free(xin);
    }
    float *rows = rand_f32((size_t)done * D, 0.f, 1.2f);
    const int t = done / 4;
#ifdef PIN_REFERENCE
    bad |= write_file(argv[1], "ref", "enc_cache_len", "i32", &ctx->enc_kv_cache_len, sizeof ctx->enc_kv_cache_len);
    int t_ref = 0;
    float *a_ref = vox_adapter_forward(ctx, rows, done, &t_ref);
    if (t_ref != t) return 4;
    bad |= write_file(argv[1], "ref", "adapter", "f32", a_ref, (size_t)t * VOX_DEC_DIM * 4);
#endif
    float *a_orc = malloc((size_t)t * VOX_DEC_DIM * 4);
    orc_adapter(a_orc, rows, done, ctx->adapter.linear0_weight_bf16, ctx->adapter.linear1_weight_bf16, D, VOX_DEC_DIM);
    bad |= write_file(argv[1], "orc", "adapter", "f32", a_orc, (size_t)t * VOX_DEC_DIM * 4);
    return bad;
}
