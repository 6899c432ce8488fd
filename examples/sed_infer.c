/* sed_infer.c -- Cnn_9layers_Gru_FrameAtt inference through the C ABI alone (no Python, no tensor library).
 *
 *   sed_infer <weights.bin> <wave.bin> <out.bin> [n_fft hop]        (defaults 512 160 = the 16 kHz preset)
 *
 * What the reference does in pytorch/models.py:625-688 (Cnn_9layers_Gru_FrameAtt.forward) on a state_dict loaded by
 * pytorch/predict.py:225-236, done by a plain C program: read the reference-layout parameters as raw float32 arrays,
 * prepare them with the sed_fold_bn / sed_pack_* helpers, run the kernels of include/sed_b200.h, write the two outputs
 * the reference callers read (clipwise_output, framewise_output).  tests/test_gpu_c_driver.py checks the result bit for
 * bit against the Python host engine on the same files.
 *
 * weights.bin: int32 count, then per tensor: int32 name_len, name, int32 ndim, int64 dims[ndim], float32 data (the
 * state_dict keys of SURVEY.md 8b).  wave.bin: int32 B, int32 L, float32 [B][L].
 * out.bin: int32 B, int32 frames, int32 classes, float32 clipwise [B][25], float32 framewise [B][frames][25].
 */
#include <math.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cuda_runtime_api.h>

#include "../include/sed_b200.h"

#define CHECK_CUDA(x)                                                                      \
  do {                                                                                     \
    cudaError_t e_ = (x);                                                                  \
    if (e_ != cudaSuccess) {                                                               \
      fprintf(stderr, "%s:%d %s: %s\n", __FILE__, __LINE__, #x, cudaGetErrorString(e_));   \
      exit(2);                                                                             \
    }                                                                                      \
  } while (0)
#define CHECK_SED(x)                                                                       \
  do {                                                                                     \
    int rc_ = (x);                                                                         \
    if (rc_ != SED_OK) {                                                                   \
      fprintf(stderr, "%s:%d %s -> %d: %s\n", __FILE__, __LINE__, #x, rc_, sed_last_error_string()); \
      exit(3);                                                                             \
    }                                                                                      \
  } while (0)

typedef struct {
  char name[96];
  int ndim;
  long dims[4];
  long numel;
  float* host;
} Tensor;

static Tensor g_tensors[128];
static int g_count = 0;

static void must_read(void* dst, size_t size, size_t n, FILE* f, const char* what) {
  if (fread(dst, size, n, f) != n) {
    fprintf(stderr, "short read: %s\n", what);
    exit(1);
  }
}

static void load_weights(const char* path) {
  FILE* f = fopen(path, "rb");
  if (!f) {
    perror(path);
    exit(1);
  }
  int32_t count;
  must_read(&count, 4, 1, f, "count");
  if (count < 1 || count > 128) {
    fprintf(stderr, "bad tensor count %d\n", count);
    exit(1);
  }
  for (int i = 0; i < count; ++i) {
    Tensor* t = &g_tensors[i];
    int32_t len, ndim;
    must_read(&len, 4, 1, f, "name length");
    if (len < 1 || len >= (int)sizeof(t->name)) {
      fprintf(stderr, "bad name length %d\n", len);
      exit(1);
    }
    must_read(t->name, 1, (size_t)len, f, "name");
    t->name[len] = 0;
    must_read(&ndim, 4, 1, f, "ndim");
    if (ndim < 0 || ndim > 4) {
      fprintf(stderr, "%s: ndim %d\n", t->name, ndim);
      exit(1);
    }
    t->ndim = ndim;
    t->numel = 1;
    for (int d = 0; d < ndim; ++d) {
      int64_t v;
      must_read(&v, 8, 1, f, "dim");
      t->dims[d] = (long)v;
      t->numel *= (long)v;
    }
    t->host = (float*)malloc(sizeof(float) * (size_t)(t->numel > 0 ? t->numel : 1));
    must_read(t->host, 4, (size_t)t->numel, f, t->name);
  }
  g_count = count;
  fclose(f);
}

static const Tensor* find(const char* name, long expect_numel) {
  for (int i = 0; i < g_count; ++i)
    if (strcmp(g_tensors[i].name, name) == 0) {
      if (expect_numel > 0 && g_tensors[i].numel != expect_numel) {
        fprintf(stderr, "%s: %ld elements, expected %ld\n", name, g_tensors[i].numel, expect_numel);
        exit(1);
      }
      return &g_tensors[i];
    }
  fprintf(stderr, "missing tensor %s\n", name);
  exit(1);
}

static void* dev_alloc(size_t bytes) {
  void* p = NULL;
  CHECK_CUDA(cudaMalloc(&p, bytes ? bytes : 16));
  return p;
}

static float* upload(const float* host, long n) {
  float* d = (float*)dev_alloc(sizeof(float) * (size_t)n);
  CHECK_CUDA(cudaMemcpy(d, host, sizeof(float) * (size_t)n, cudaMemcpyHostToDevice));
  return d;
}

static float* upload_named(const char* name, long expect) { return upload(find(name, expect)->host, find(name, expect)->numel); }

/* eval-mode BatchNorm `prefix` folded to scale / shift [n] on the device */
static void fold(const char* prefix, int n, float** scale, float** shift) {
  char key[128];
  float* raw[4];
  const char* parts[4] = {".weight", ".bias", ".running_mean", ".running_var"};
  for (int k = 0; k < 4; ++k) {
    snprintf(key, sizeof(key), "%s%s", prefix, parts[k]);
    raw[k] = upload_named(key, n);
  }
  *scale = (float*)dev_alloc(sizeof(float) * (size_t)n);
  *shift = (float*)dev_alloc(sizeof(float) * (size_t)n);
  CHECK_SED(sed_fold_bn(raw[0], raw[1], raw[2], raw[3], n, 1e-5, *scale, *shift, NULL));
  CHECK_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 4; ++k) cudaFree(raw[k]);
}

int main(int argc, char** argv) {
  if (argc < 4) {
    fprintf(stderr, "usage: %s weights.bin wave.bin out.bin [n_fft hop]\n", argv[0]);
    return 1;
  }
  const int n_fft = argc > 4 ? atoi(argv[4]) : 512;
  const int hop = argc > 5 ? atoi(argv[5]) : 160;
  const int F = n_fft / 2 + 1, M = 64, DT = SED_DTYPE_F16;
  if (sed_abi_version() != 13) {
    fprintf(stderr, "libsed_b200 ABI %d, this driver was written against 13\n", sed_abi_version());
    return 1;
  }
  load_weights(argv[1]);

  /* ---- waveform ---- */
  FILE* fw = fopen(argv[2], "rb");
  if (!fw) {
    perror(argv[2]);
    return 1;
  }
  int32_t B, L;
  must_read(&B, 4, 1, fw, "B");
  must_read(&L, 4, 1, fw, "L");
  float* wave_h = (float*)malloc(sizeof(float) * (size_t)B * (size_t)L);
  must_read(wave_h, 4, (size_t)B * (size_t)L, fw, "waveform");
  fclose(fw);
  float* wave = upload(wave_h, (long)B * L);
  const int T = L / hop + 1, H1 = T / 2, H2 = T / 4, Tp = T / 8;
  if (Tp < 1) {
    fprintf(stderr, "clip too short\n");
    return 1;
  }
  const int Bp = (B + 127) / 128 * 128;

  /* ---- front-end constants (stft.py:192-212: the window is row 0 of conv_real; stft.py:688: melW) ---- */
  const Tensor* conv_real = find("spectrogram_extractor.stft.conv_real.weight", (long)F * n_fft);
  float* window = upload(conv_real->host, n_fft);
  float* tw_h = (float*)malloc(sizeof(float) * 2 * (size_t)n_fft);
  CHECK_SED(sed_frontend_twiddle(n_fft, tw_h));
  float* twiddle = upload(tw_h, 2L * n_fft);
  const Tensor* melW = find("logmel_extractor.melW", (long)F * M);
  int lo_h[64], len_h[64], off_h[64], n_val = 0;
  float* val_h = (float*)malloc(sizeof(float) * (size_t)F * M);
  CHECK_SED(sed_band_mel(melW->host, F, M, lo_h, len_h, off_h, val_h, F * M, &n_val));
  int *mel_lo = (int*)dev_alloc(sizeof(lo_h)), *mel_len = (int*)dev_alloc(sizeof(len_h)), *mel_off = (int*)dev_alloc(sizeof(off_h));
  CHECK_CUDA(cudaMemcpy(mel_lo, lo_h, sizeof(lo_h), cudaMemcpyHostToDevice));
  CHECK_CUDA(cudaMemcpy(mel_len, len_h, sizeof(len_h), cudaMemcpyHostToDevice));
  CHECK_CUDA(cudaMemcpy(mel_off, off_h, sizeof(off_h), cudaMemcpyHostToDevice));
  float* mel_val = upload(val_h, n_val > 0 ? n_val : 1);
  const float amin = 1e-10f;
  const float db_offset = (float)(10.0 * log10(fmax((double)amin, 1.0))); /* ref = 1.0, models.py:572 */

  /* ---- weights ---- */
  float *bn0_s, *bn0_b, *c11_s, *c11_b;
  fold("bn0", 64, &bn0_s, &bn0_b);
  fold("conv_block1.bn1", 64, &c11_s, &c11_b);
  float* w1 = upload_named("conv_block1.conv1.weight", 64 * 9);
  float* w1_scaled = (float*)dev_alloc(sizeof(float) * 64 * 9);
  CHECK_SED(sed_pack_conv_first(w1, c11_s, w1_scaled, NULL));
  static const struct { const char* conv; const char* bn; int cin, cout, mode; } layers[7] = {
      {"conv_block1.conv2.weight", "conv_block1.bn2", 64, 64, SED_CONV_POOL},
      {"conv_block2.conv1.weight", "conv_block2.bn1", 64, 128, SED_CONV_STORE},
      {"conv_block2.conv2.weight", "conv_block2.bn2", 128, 128, SED_CONV_POOL},
      {"conv_block3.conv1.weight", "conv_block3.bn1", 128, 256, SED_CONV_STORE},
      {"conv_block3.conv2.weight", "conv_block3.bn2", 256, 256, SED_CONV_POOL},
      {"conv_block4.conv1.weight", "conv_block4.bn1", 256, 512, SED_CONV_STORE},
      {"conv_block4.conv2.weight", "conv_block4.bn2", 512, 512, SED_CONV_FREQMEAN}};
  void* wp[7];
  float *cs[7], *cb[7];
  for (int i = 0; i < 7; ++i) {
    const long n = (long)layers[i].cout * layers[i].cin * 9;
    float* w = upload_named(layers[i].conv, n);
    wp[i] = dev_alloc(2 * (size_t)n);
    CHECK_SED(sed_pack_conv3x3(w, layers[i].cout, layers[i].cin, wp[i], DT, NULL));
    CHECK_CUDA(cudaDeviceSynchronize());
    cudaFree(w);
    fold(layers[i].bn, layers[i].cout, &cs[i], &cb[i]);
  }
  /* nn.GRU parameters (models.py:614-615): forward and reverse direction stacked */
  float* wih32 = (float*)dev_alloc(sizeof(float) * 1536 * 512);
  CHECK_CUDA(cudaMemcpy(wih32, find("gru.weight_ih_l0", 768 * 512)->host, sizeof(float) * 768 * 512, cudaMemcpyHostToDevice));
  CHECK_CUDA(cudaMemcpy(wih32 + 768 * 512, find("gru.weight_ih_l0_reverse", 768 * 512)->host, sizeof(float) * 768 * 512,
                        cudaMemcpyHostToDevice));
  void* wih16 = dev_alloc(2 * 1536 * 512);
  CHECK_SED(sed_cast_16(wih32, 1536L * 512, wih16, DT, NULL));
  float* bih = (float*)dev_alloc(sizeof(float) * 1536);
  CHECK_CUDA(cudaMemcpy(bih, find("gru.bias_ih_l0", 768)->host, sizeof(float) * 768, cudaMemcpyHostToDevice));
  CHECK_CUDA(cudaMemcpy(bih + 768, find("gru.bias_ih_l0_reverse", 768)->host, sizeof(float) * 768, cudaMemcpyHostToDevice));
  float* bhh = (float*)dev_alloc(sizeof(float) * 1536);
  CHECK_CUDA(cudaMemcpy(bhh, find("gru.bias_hh_l0", 768)->host, sizeof(float) * 768, cudaMemcpyHostToDevice));
  CHECK_CUDA(cudaMemcpy(bhh + 768, find("gru.bias_hh_l0_reverse", 768)->host, sizeof(float) * 768, cudaMemcpyHostToDevice));
  float* whh_f = upload_named("gru.weight_hh_l0", 768 * 256);
  float* whh_r = upload_named("gru.weight_hh_l0_reverse", 768 * 256);
  void* whh16 = dev_alloc(2 * 1536 * 256);
  CHECK_SED(sed_pack_gru_whh(whh_f, whh_r, whh16, DT, NULL));
  float* w_att = upload_named("att_block.att.weight", 25 * 512);
  float* b_att = upload_named("att_block.att.bias", 25);
  float* w_cla = upload_named("att_block.cla.weight", 25 * 512);
  float* b_cla = upload_named("att_block.cla.bias", 25);

  /* ---- activations (SURVEY.md 8a: NHWC 16-bit, features time-major over the batch padded to 128 clips) ---- */
  float* logmel = (float*)dev_alloc(sizeof(float) * (size_t)B * T * 64);
  void* p1 = dev_alloc(2 * (size_t)B * H1 * 32 * 64);
  void* a2 = dev_alloc(2 * (size_t)B * H1 * 32 * 128);
  void* p2 = dev_alloc(2 * (size_t)B * H2 * 16 * 128);
  void* a3 = dev_alloc(2 * (size_t)B * H2 * 16 * 256);
  void* p3 = dev_alloc(2 * (size_t)B * Tp * 8 * 256);
  void* a4 = dev_alloc(2 * (size_t)B * Tp * 8 * 512);
  const size_t feat_bytes = 2 * (size_t)Tp * Bp * 512;
  void* feat = dev_alloc(feat_bytes);
  CHECK_CUDA(cudaMemset(feat, 0, feat_bytes)); /* rows of padding clips */
  float* gi = (float*)dev_alloc(sizeof(float) * (size_t)Tp * Bp * 1536);
  float* gru_out = (float*)dev_alloc(sizeof(float) * (size_t)Tp * Bp * 512);
  void* gru_ws = dev_alloc((size_t)sed_bigru_workspace_bytes(B));
  void* scratch = dev_alloc((size_t)sed_attpool_blocks_scratch_bytes(B, Tp));
  int frames = Tp * 8; /* interpolate x8, then pad to 100-frame blocks unless 1000 (models.py:62-63, 677-681) */
  if (frames != 1000 && frames % 100) frames += 100 - frames % 100;
  float* clip = (float*)dev_alloc(sizeof(float) * (size_t)B * 25);
  float* frame = (float*)dev_alloc(sizeof(float) * (size_t)B * frames * 25);

  /* ---- the forward pass: every call is asynchronous on the (default) stream ---- */
  CHECK_SED(sed_frontend_logmel(wave, 0, B, L, L, NULL, (long)B * L, n_fft, hop, window, twiddle, mel_lo, mel_len, mel_off,
                                mel_val, M, amin, db_offset, 1, bn0_s, bn0_b, logmel, NULL));
  CHECK_SED(sed_conv_block1(logmel, B, T, 64, w1_scaled, c11_b, wp[0], cs[0], cb[0], p1, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(p1, B, H1, 32, 64, wp[1], cs[1], cb[1], 128, SED_CONV_STORE, a2, NULL, 0, 0, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(a2, B, H1, 32, 128, wp[2], cs[2], cb[2], 128, SED_CONV_POOL, p2, NULL, 0, 0, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(p2, B, H2, 16, 128, wp[3], cs[3], cb[3], 256, SED_CONV_STORE, a3, NULL, 0, 0, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(a3, B, H2, 16, 256, wp[4], cs[4], cb[4], 256, SED_CONV_POOL, p3, NULL, 0, 0, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(p3, B, Tp, 8, 256, wp[5], cs[5], cb[5], 512, SED_CONV_STORE, a4, NULL, 0, 0, DT, NULL));
  CHECK_SED(sed_conv3x3_bn_relu(a4, B, Tp, 8, 512, wp[6], cs[6], cb[6], 512, SED_CONV_FREQMEAN, feat, NULL, 1, Bp, DT,
                                NULL));
  CHECK_SED(sed_linear(feat, (long)Tp * Bp, 512, wih16, bih, 1536, 0, gi, NULL, 1, DT, NULL));
  CHECK_SED(sed_bigru(gi, whh16, bhh, B, Tp, gru_out, gru_ws, DT, NULL));
  CHECK_SED(sed_attpool_blocks(gru_out, B, Tp, w_att, b_att, w_cla, b_cla, 8, frames, scratch, clip, frame, NULL, NULL, 0,
                               0, B, NULL));
  CHECK_CUDA(cudaDeviceSynchronize());

  /* ---- results ---- */
  float* clip_h = (float*)malloc(sizeof(float) * (size_t)B * 25);
  float* frame_h = (float*)malloc(sizeof(float) * (size_t)B * frames * 25);
  CHECK_CUDA(cudaMemcpy(clip_h, clip, sizeof(float) * (size_t)B * 25, cudaMemcpyDeviceToHost));
  CHECK_CUDA(cudaMemcpy(frame_h, frame, sizeof(float) * (size_t)B * frames * 25, cudaMemcpyDeviceToHost));
  FILE* fo = fopen(argv[3], "wb");
  if (!fo) {
    perror(argv[3]);
    return 1;
  }
  const int32_t hdr[3] = {B, frames, 25};
  fwrite(hdr, 4, 3, fo);
  fwrite(clip_h, 4, (size_t)B * 25, fo);
  fwrite(frame_h, 4, (size_t)B * frames * 25, fo);
  fclose(fo);
  printf("sed_infer: %d clips x %d samples -> clipwise [%d,25], framewise [%d,%d,25]; clip[0][0..2] = %.6f %.6f %.6f\n", B, L,
         B, B, frames, clip_h[0], clip_h[1], clip_h[2]);
  return 0;
}
