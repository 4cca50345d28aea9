/* raft_flow.c -- the whole RAFT call of librdvc_corr.so from plain C: pack a raft_large state dict, run
 * rdvc_corr_raft_flow_sequence on a few frames at 368x640 (RDVC's RAFT size, R:codec_processing.py:649-650) and write the
 * flows to a file.  No PyTorch; the CUDA runtime only allocates and copies.
 *
 *   gcc -std=c99 -Iinclude -I/usr/local/cuda/include examples/raft_flow.c -o raft_flow \
 *       -L<pkg>/lib -lrdvc_corr -Wl,-rpath,<pkg>/lib -L/usr/local/cuda/lib64 -lcudart -lm
 *   ./raft_flow flows.f32 [state.bin]
 *
 * state.bin (optional; without it the weights are generated from a fixed seed): a uint32 count, then per tensor a
 * uint32 name length, the name, a uint32 ndim, ndim int64 dims and the fp32 values, little-endian.  The frames are
 * N_FRAMES moving integer patterns / 255 in fp32, NCHW.  flows.f32: (N_FRAMES - 1, 2, 368, 640) fp32 values. */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "rdvc_corr.h"

#define N_FRAMES 3
#define H 368
#define W 640
#define ITERS 12

typedef struct {
    char name[96];
    int ndim;
    long long shape[4];
    float* data;
} Tensor;

static Tensor* g_t;
static int g_n;
static uint64_t g_rng = 0x9E3779B97F4A7C15ull;

static float uniform(float a) {            /* xorshift64*: uniform in [-a, a) */
    g_rng ^= g_rng >> 12; g_rng ^= g_rng << 25; g_rng ^= g_rng >> 27;
    return a * ((float)((g_rng * 0x2545F4914F6CDD1Dull) >> 40) / 8388608.0f - 1.0f);
}

static long long numel(const Tensor* t) {
    long long n = 1;
    for (int i = 0; i < t->ndim; ++i) n *= t->shape[i];
    return n;
}

/* one tensor of the generated state dict: kind 0 = weight (scale 1/sqrt(fan in)), 1 = bias, 2 = BN scale, 3 = BN var */
static void add(const char* name, int ndim, long long d0, long long d1, long long d2, long long d3, int kind, float fan) {
    Tensor* t = &g_t[g_n++];
    snprintf(t->name, sizeof t->name, "%s", name);
    t->ndim = ndim;
    t->shape[0] = d0; t->shape[1] = d1; t->shape[2] = d2; t->shape[3] = d3;
    t->data = (float*)malloc(sizeof(float) * (size_t)numel(t));
    for (long long i = 0; i < numel(t); ++i)
        t->data[i] = kind == 0 ? uniform(1.0f / fan) : kind == 1 ? uniform(0.05f)
                     : kind == 2 ? 1.0f + uniform(0.1f) : 1.0f + uniform(0.5f);
}

static void conv(const char* prefix, int cout, int cin, int kh, int kw) {
    char n[96];
    snprintf(n, sizeof n, "%s.weight", prefix);
    add(n, 4, cout, cin, kh, kw, 0, sqrtf((float)(cin * kh * kw)));
    snprintf(n, sizeof n, "%s.bias", prefix);
    add(n, 1, cout, 1, 1, 1, 1, 0);
}

static void generate(void) {
    static const struct { const char* name; int cout, cin, k; } enc[16] = {
        {"convnormrelu", 64, 3, 7}, {"layer1.0.convnormrelu1", 64, 64, 3}, {"layer1.0.convnormrelu2", 64, 64, 3},
        {"layer1.1.convnormrelu1", 64, 64, 3}, {"layer1.1.convnormrelu2", 64, 64, 3},
        {"layer2.0.convnormrelu1", 96, 64, 3}, {"layer2.0.downsample", 96, 64, 1}, {"layer2.0.convnormrelu2", 96, 96, 3},
        {"layer2.1.convnormrelu1", 96, 96, 3}, {"layer2.1.convnormrelu2", 96, 96, 3},
        {"layer3.0.convnormrelu1", 128, 96, 3}, {"layer3.0.downsample", 128, 96, 1},
        {"layer3.0.convnormrelu2", 128, 128, 3}, {"layer3.1.convnormrelu1", 128, 128, 3},
        {"layer3.1.convnormrelu2", 128, 128, 3}, {"conv", 256, 128, 1}};
    char n[96];
    g_t = (Tensor*)calloc(256, sizeof(Tensor));
    for (int e = 0; e < 2; ++e)
        for (int i = 0; i < 16; ++i) {
            const char* pre = e ? "context_encoder" : "feature_encoder";
            snprintf(n, sizeof n, "%s.%s%s", pre, enc[i].name, i < 15 ? ".0" : "");
            conv(n, enc[i].cout, enc[i].cin, enc[i].k, enc[i].k);
            if (e && i < 15) {                 /* BatchNorm2d: weight, bias, running_mean, running_var */
                static const char* bn[4] = {"weight", "bias", "running_mean", "running_var"};
                static const int kinds[4] = {2, 1, 1, 3};
                for (int j = 0; j < 4; ++j) {
                    snprintf(n, sizeof n, "%s.%s.1.%s", pre, enc[i].name, bn[j]);
                    add(n, 1, enc[i].cout, 1, 1, 1, kinds[j], 0);
                }
            }
        }
    conv("update_block.motion_encoder.convcorr1.0", 256, 324, 1, 1);
    conv("update_block.motion_encoder.convcorr2.0", 192, 256, 3, 3);
    conv("update_block.motion_encoder.convflow1.0", 128, 2, 7, 7);
    conv("update_block.motion_encoder.convflow2.0", 64, 128, 3, 3);
    conv("update_block.motion_encoder.conv.0", 126, 256, 3, 3);
    for (int g = 1; g <= 2; ++g)
        for (int q = 0; q < 3; ++q) {
            snprintf(n, sizeof n, "update_block.recurrent_block.convgru%d.conv%c", g, "zrq"[q]);
            conv(n, 128, 384, g == 1 ? 1 : 5, g == 1 ? 5 : 1);
        }
    conv("update_block.flow_head.conv1", 256, 128, 3, 3);
    conv("update_block.flow_head.conv2", 2, 256, 3, 3);
    conv("mask_predictor.convrelu.0", 256, 128, 3, 3);
    conv("mask_predictor.conv", 576, 256, 1, 1);
}

static int load(const char* path) {
    FILE* f = fopen(path, "rb");
    uint32_t n = 0;
    if (!f || fread(&n, 4, 1, f) != 1 || n > 4096) return 1;
    g_t = (Tensor*)calloc(n, sizeof(Tensor));
    for (uint32_t i = 0; i < n; ++i) {
        Tensor* t = &g_t[g_n++];
        uint32_t len = 0, nd = 0;
        if (fread(&len, 4, 1, f) != 1 || len >= sizeof t->name || fread(t->name, 1, len, f) != len) return 1;
        if (fread(&nd, 4, 1, f) != 1 || nd > 4 || fread(t->shape, 8, nd, f) != nd) return 1;
        t->ndim = (int)nd;
        t->data = (float*)malloc(sizeof(float) * (size_t)numel(t) + 1);
        if (fread(t->data, 4, (size_t)numel(t), f) != (size_t)numel(t)) return 1;
    }
    fclose(f);
    return 0;
}

#define CUDA_OK(x) do { cudaError_t e_ = (x); if (e_ != cudaSuccess) { \
    fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_)); return 1; } } while (0)

int main(int argc, char** argv) {
    if (argc < 2) {
        fprintf(stderr, "usage: %s flows.f32 [state.bin]\n", argv[0]);
        return 2;
    }
    if (argc > 2 ? load(argv[2]) : (generate(), 0)) {
        fprintf(stderr, "cannot read %s\n", argv[2]);
        return 1;
    }
    /* 1. pack on the host, copy to the device */
    const char** names = (const char**)malloc(sizeof(char*) * g_n);
    const float** data = (const float**)malloc(sizeof(float*) * g_n);
    int* ndims = (int*)malloc(sizeof(int) * g_n);
    const long long** shapes = (const long long**)malloc(sizeof(long long*) * g_n);
    for (int i = 0; i < g_n; ++i) {
        names[i] = g_t[i].name; data[i] = g_t[i].data; ndims[i] = g_t[i].ndim; shapes[i] = g_t[i].shape;
    }
    const size_t wbytes = rdvc_corr_raft_packed_weight_bytes(RDVC_DT_F16);
    void* packed = malloc(wbytes);
    int rc = rdvc_corr_raft_pack_weights(names, data, ndims, shapes, g_n, RDVC_DT_F16, packed, wbytes);
    if (rc != RDVC_OK) {
        fprintf(stderr, "rdvc_corr_raft_pack_weights failed (%d): %s\n", rc, rdvc_corr_last_error());
        return 1;
    }
    /* 2. frames: a texture moving by (2, 1) pixels per frame */
    const size_t plane = (size_t)H * W, fbytes = sizeof(float) * N_FRAMES * 3 * plane;
    float* frames = (float*)malloc(fbytes);
    for (int f = 0; f < N_FRAMES; ++f)
        for (int c = 0; c < 3; ++c)
            for (int y = 0; y < H; ++y)
                for (int x = 0; x < W; ++x) {
                    const int u = x - 2 * f + 64, v = y - f + 64;
                    frames[((size_t)f * 3 + c) * plane + (size_t)y * W + x] =
                        (float)((u * 7 + v * 13 + (u / 16) * (v / 16) * 29 + c * 31) % 256) / 255.0f;
                }
    const size_t ws_bytes = rdvc_corr_raft_workspace_bytes(N_FRAMES, N_FRAMES - 1, H, W, RDVC_DT_F16, RDVC_DT_F32);
    const size_t out_bytes = sizeof(float) * (N_FRAMES - 1) * 2 * plane;
    void *d_w, *d_frames, *d_ws, *d_out;
    cudaStream_t st;
    CUDA_OK(cudaMalloc(&d_w, wbytes));
    CUDA_OK(cudaMalloc(&d_frames, fbytes));
    CUDA_OK(cudaMalloc(&d_ws, ws_bytes));
    CUDA_OK(cudaMalloc(&d_out, out_bytes));
    CUDA_OK(cudaStreamCreate(&st));
    CUDA_OK(cudaMemcpy(d_w, packed, wbytes, cudaMemcpyHostToDevice));
    CUDA_OK(cudaMemcpyAsync(d_frames, frames, fbytes, cudaMemcpyHostToDevice, st));
    /* 3. the whole call: fp16 activations (the reference's GPU default), fp32 correlation volume */
    const long long strides[4] = {3 * (long long)plane, (long long)plane, W, 1};
    rc = rdvc_corr_raft_flow_sequence(d_frames, strides, RDVC_DT_F32, N_FRAMES, H, W, ITERS, RDVC_DT_F16, RDVC_DT_F32, d_w, 0.25f,
                                 d_ws, ws_bytes, (float*)d_out, st);
    if (rc != RDVC_OK) {
        fprintf(stderr, "rdvc_corr_raft_flow_sequence failed (%d): %s\n", rc, rdvc_corr_last_error());
        return 1;
    }
    float* out = (float*)malloc(out_bytes);
    CUDA_OK(cudaMemcpyAsync(out, d_out, out_bytes, cudaMemcpyDeviceToHost, st));
    CUDA_OK(cudaStreamSynchronize(st));
    /* 4. write the flows */
    FILE* f = fopen(argv[1], "wb");
    if (!f || fwrite(out, 1, out_bytes, f) != out_bytes || fclose(f)) {
        fprintf(stderr, "cannot write %s\n", argv[1]);
        return 1;
    }
    double s = 0.0;
    for (size_t i = 0; i < out_bytes / sizeof(float); ++i) s += out[i] < 0 ? -out[i] : out[i];
    printf("%d flows of %dx%d written to %s, mean |flow| = %.4f px\n", N_FRAMES - 1, H, W, argv[1],
           s / (double)(out_bytes / sizeof(float)));
    cudaStreamDestroy(st);
    cudaFree(d_w); cudaFree(d_frames); cudaFree(d_ws); cudaFree(d_out);
    for (int i = 0; i < g_n; ++i) free(g_t[i].data);
    free(g_t); free(names); free(data); free(ndims); free(shapes); free(packed); free(frames); free(out);
    return 0;
}
