// xvb-extract: Python-free x-vector extraction over the C ABI (SURVEY section 8f rank 4).
//
//   xvb-extract [--batch N] [--max-chunk N] [--ragged] [--cmn none|utt|sliding] [--cmn-window W] [--gpu-id ID]
//               [--wav fbank|mfcc [--num-mel-bins N] [--num-ceps N] [--low-freq F] [--high-freq F]
//                [--frame-length MS] [--frame-shift MS] [--energy-floor E] [--use-energy]]
//               <model.xvbm> <feats-rspecifier | wav.scp> <vectors-wspecifier>
//
// With --wav the second positional is a Kaldi wav.scp (`<key> <file.wav>`, PCM16 RIFF; samples are used
// in int16 range like runtime/frontend/wav.h:95-99 and processor.py:429) and features are computed on
// the GPU by xvb_fbank_compute with the given kaldi_featset (runtime/test/feat_conf.yaml names); add
// `--cmn utt` for that file's `mean_norm: true`.
//
// Positionals follow the reference's extractor CLI (pytorch/pipeline/onestep/extract_embeddings.py
// :17-45: <model-path> <feats-rspecifier> <vectors-wspecifier>); the role is that of the reference's
// C++ runtime (runtime/bin/extractor_main.cc + runtime/extractor/torch_asv_extractor.cc:71-122: load
// a model, optional per-utterance CMN, extract, emit the vector), with features instead of wav on
// the input side.  What it adds: utterances of equal length are batched (the reference runs batch 1).
//   * chunk rule of framework.py:34-47: T > max-chunk -> num_split = ceil(T/max), split = T/num_split,
//     the last chunk takes the remainder, embedding = sum(len_i * emb_i) / T in fp32;
//   * one "FV" vector per input key (order follows batch completion, which the wspecifier allows);
//   * --ragged (TDNN x-vector models): instead of exact-length buckets, the chunks of a window of utterances (up to
//     4 M frames) go through ONE xvb_extractor_extract_ragged_shard_host call -- length-sorted batches of mixed
//     lengths, each chunk computed as if alone -- and the vectors are written in input order;
//   * errors: message with "ERROR" on stderr, exit status 1 (the reference's shell greps for it,
//     extract_xvectors_for_pytorch.sh:144-145).  No GPU / not a B200 -> error, there is no CPU path.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "../../include/xvb200.h"

namespace {

struct Item {          // one chunk of one utterance
  int utt;
  int frames;
  std::vector<float> feats;   // (frames, F)
};

struct Utt {
  std::string key;
  int frames = 0;
  int pending = 0;            // chunks not yet extracted
  std::vector<float> acc;     // sum(len_i * emb_i)
};

[[noreturn]] void die(const char* what) {
  const char* e = xvb_last_error();
  fprintf(stderr, "ERROR: xvb-extract: %s%s%s\n", what, (e && e[0]) ? ": " : "", (e && e[0]) ? e : "");
  exit(1);
}

#define CK(call, what) do { if ((call) != XVB_OK) die(what); } while (0)
#define CU(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) { fprintf(stderr, "ERROR: xvb-extract: %s: %s\n", #call, cudaGetErrorString(_e)); exit(1); } } while (0)

struct Runner {
  xvb_extractor_t* ex = nullptr;   // TDNN x-vector family (XVBM0001) ...
  xvb_ecapa_t* ec = nullptr;       // ... or ECAPA-TDNN (XVBE0001)
  xvb_ark_writer_t* out = nullptr;
  int F = 0, D = 0, batch = 256, cmn = 0, cmn_window = 300;
  float *d_feats = nullptr, *d_tmp = nullptr, *d_emb = nullptr, *h_feats = nullptr, *h_emb = nullptr;
  float* h_ragged = nullptr;   // --ragged: a window's chunks back to back, pinned
  size_t ragged_cap = 0;
  int32_t* d_off = nullptr;
  size_t cap_frames = 0;
  std::vector<Utt> utts;
  long done_utts = 0, done_frames = 0;

  void reserve(size_t frames) {
    if (frames <= cap_frames) return;
    if (d_feats) { cudaFree(d_feats); cudaFree(d_tmp); cudaFreeHost(h_feats); }
    cap_frames = frames + frames / 4;
    CU(cudaMalloc(&d_feats, cap_frames * F * sizeof(float)));
    CU(cudaMalloc(&d_tmp, cap_frames * F * sizeof(float)));
    CU(cudaMallocHost(&h_feats, cap_frames * F * sizeof(float)));
  }

  // per-utterance / sliding CMN of whole utterances laid back to back on the device (frontend.cu)
  void cmn_device(float* x, float* y, const std::vector<int32_t>& off) {
    CU(cudaMemcpy(d_off, off.data(), off.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    CK(xvb_cmn(x, d_off, (int)off.size() - 1, F, cmn == 2 ? cmn_window : 0, y, nullptr), "xvb_cmn");
  }

  void run(std::vector<Item>& items) {
    if (items.empty()) return;
    const int B = (int)items.size(), T = items[0].frames;
    reserve((size_t)B * T);
    for (int i = 0; i < B; ++i) memcpy(h_feats + (size_t)i * T * F, items[i].feats.data(), (size_t)T * F * sizeof(float));
    CU(cudaMemcpy(d_feats, h_feats, (size_t)B * T * F * sizeof(float), cudaMemcpyHostToDevice));
    if (ex) CK(xvb_extractor_extract(ex, d_feats, B, T, d_emb, nullptr), "xvb_extractor_extract");
    else CK(xvb_ecapa_extract(ec, d_feats, B, T, d_emb, nullptr), "xvb_ecapa_extract");
    CU(cudaMemcpy(h_emb, d_emb, (size_t)B * D * sizeof(float), cudaMemcpyDeviceToHost));
    for (int i = 0; i < B; ++i) accumulate(items[i], h_emb + (size_t)i * D);
    items.clear();
  }

  // --ragged: the window's chunks in one shard call; results come back in window order
  void run_ragged(std::vector<Item>& items) {
    if (items.empty()) return;
    const int64_t n = (int64_t)items.size();
    std::vector<int64_t> off((size_t)n + 1, 0);
    for (int64_t i = 0; i < n; ++i) off[i + 1] = off[i] + items[i].frames;
    if ((size_t)off[n] > ragged_cap) {
      if (h_ragged) cudaFreeHost(h_ragged);
      ragged_cap = (size_t)off[n] + (size_t)off[n] / 4;
      CU(cudaMallocHost(&h_ragged, ragged_cap * F * sizeof(float)));
    }
    for (int64_t i = 0; i < n; ++i) memcpy(h_ragged + (size_t)off[i] * F, items[i].feats.data(), (size_t)items[i].frames * F * sizeof(float));
    std::vector<float> emb((size_t)n * D);
    CK(xvb_extractor_extract_ragged_shard_host(ex, h_ragged, off.data(), n, batch, 0, emb.data(), nullptr),
       "xvb_extractor_extract_ragged_shard_host");
    for (int64_t i = 0; i < n; ++i) accumulate(items[i], emb.data() + (size_t)i * D);
    items.clear();
  }

  // chunk rule: sum(len_i * emb_i) / T, the vector is written when the utterance's last chunk is in
  void accumulate(const Item& it, const float* e) {
    Utt& u = utts[it.utt];
    const float len = (float)it.frames;
    if (u.acc.empty()) u.acc.assign(D, 0.f);
    for (int d = 0; d < D; ++d) u.acc[d] += len * e[d];
    if (--u.pending == 0) {
      const float total = (float)u.frames;
      for (int d = 0; d < D; ++d) u.acc[d] /= total;
      CK(xvb_ark_writer_put_vector(out, u.key.c_str(), u.acc.data(), D), "writing a vector");
      std::vector<float>().swap(u.acc);
      ++done_utts;
      done_frames += u.frames;
    }
  }
};

// PCM16 RIFF reader: channel 0 as float in int16 range (runtime/frontend/wav.h:44-118)
bool read_wav(const std::string& path, std::vector<float>* out, int* sample_rate) {
  FILE* f = fopen(path.c_str(), "rb");
  if (!f) { fprintf(stderr, "ERROR: xvb-extract: cannot open wav '%s'\n", path.c_str()); return false; }
  unsigned char hd[12];
  bool ok = fread(hd, 1, 12, f) == 12 && memcmp(hd, "RIFF", 4) == 0 && memcmp(hd + 8, "WAVE", 4) == 0;
  int channels = 0, bits = 0, fmt = 0;
  *sample_rate = 0;
  while (ok) {
    unsigned char ch[8];
    if (fread(ch, 1, 8, f) != 8) { ok = false; break; }
    const uint32_t sz = ch[4] | (ch[5] << 8) | (ch[6] << 16) | ((uint32_t)ch[7] << 24);
    if (memcmp(ch, "fmt ", 4) == 0) {
      unsigned char b[16];
      if (sz < 16 || fread(b, 1, 16, f) != 16) { ok = false; break; }
      fmt = b[0] | (b[1] << 8); channels = b[2] | (b[3] << 8);
      *sample_rate = b[4] | (b[5] << 8) | (b[6] << 16) | ((uint32_t)b[7] << 24);
      bits = b[14] | (b[15] << 8);
      fseek(f, (long)(sz - 16 + (sz & 1)), SEEK_CUR);
    } else if (memcmp(ch, "data", 4) == 0) {
      if (fmt != 1 || bits != 16 || channels < 1) { ok = false; break; }
      std::vector<int16_t> raw(sz / 2);
      const size_t got = fread(raw.data(), 2, raw.size(), f);   // a streamed header may overstate the size
      const size_t n = got / channels;
      out->resize(n);
      for (size_t i = 0; i < n; ++i) (*out)[i] = (float)raw[i * channels];
      fclose(f);
      return true;
    } else {
      fseek(f, (long)(sz + (sz & 1)), SEEK_CUR);
    }
  }
  fclose(f);
  fprintf(stderr, "ERROR: xvb-extract: '%s' is not a PCM16 RIFF wav\n", path.c_str());
  return false;
}

}  // namespace

int main(int argc, char** argv) {
  Runner r;
  int max_chunk = 10000, gpu = 0;
  bool ragged = false;
  std::string wav_type;
  xvb_fbank_opts_t fo;
  xvb_fbank_default_opts(&fo);
  bool ceps_set = false;
  std::vector<const char*> pos;
  for (int i = 1; i < argc; ++i) {
    const std::string a = argv[i];
    auto val = [&](const char* name) -> const char* {
      if (i + 1 >= argc) { fprintf(stderr, "ERROR: xvb-extract: %s needs a value\n", name); exit(1); }
      return argv[++i];
    };
    if (a == "--batch") r.batch = atoi(val("--batch"));
    else if (a == "--ragged") ragged = true;
    else if (a == "--max-chunk") max_chunk = atoi(val("--max-chunk"));
    else if (a == "--cmn-window") r.cmn_window = atoi(val("--cmn-window"));
    else if (a == "--gpu-id") gpu = atoi(val("--gpu-id"));
    else if (a == "--wav") wav_type = val("--wav");
    else if (a == "--num-mel-bins") fo.num_mel_bins = atoi(val("--num-mel-bins"));
    else if (a == "--num-ceps") { fo.num_ceps = atoi(val("--num-ceps")); ceps_set = true; }
    else if (a == "--low-freq") fo.low_freq = (float)atof(val("--low-freq"));
    else if (a == "--high-freq") fo.high_freq = (float)atof(val("--high-freq"));
    else if (a == "--frame-length") fo.frame_length_ms = (float)atof(val("--frame-length"));
    else if (a == "--frame-shift") fo.frame_shift_ms = (float)atof(val("--frame-shift"));
    else if (a == "--energy-floor") fo.energy_floor = (float)atof(val("--energy-floor"));
    else if (a == "--use-energy") fo.use_energy = 1;
    else if (a == "--cmn") {
      const std::string m = val("--cmn");
      r.cmn = m == "none" ? 0 : m == "utt" ? 1 : m == "sliding" ? 2 : -1;
      if (r.cmn < 0) { fprintf(stderr, "ERROR: xvb-extract: --cmn must be none, utt or sliding\n"); return 1; }
    } else if (a == "--help" || a == "-h") {
      printf("usage: xvb-extract [--batch N] [--max-chunk N] [--ragged] [--cmn none|utt|sliding] [--cmn-window W] [--gpu-id ID]\n"
             "                   [--wav fbank|mfcc [--num-mel-bins N] [--num-ceps N] [--low-freq F] [--high-freq F]\n"
             "                    [--frame-length MS] [--frame-shift MS] [--energy-floor E] [--use-energy]]\n"
             "                   <model.xvbm> <feats-rspecifier | wav.scp> <vectors-wspecifier>\n");
      return 0;
    } else if (a.size() > 2 && a[0] == '-' && a[1] == '-') {
      fprintf(stderr, "ERROR: xvb-extract: unknown option %s\n", a.c_str());
      return 1;
    } else pos.push_back(argv[i]);
  }
  if (!wav_type.empty() && wav_type != "fbank" && wav_type != "mfcc") { fprintf(stderr, "ERROR: xvb-extract: --wav must be fbank or mfcc\n"); return 1; }
  if (wav_type == "mfcc" && !ceps_set) fo.num_ceps = 13;
  if (wav_type == "fbank") fo.num_ceps = 0;
  if (pos.size() != 3 || r.batch < 1 || max_chunk < 1 || r.cmn_window < 1) {
    fprintf(stderr, "ERROR: xvb-extract: expected <model.xvbm> <feats-rspecifier> <vectors-wspecifier> (see --help)\n");
    return 1;
  }
  if (cudaSetDevice(gpu) != cudaSuccess) { fprintf(stderr, "ERROR: xvb-extract: no CUDA device %d visible (there is no CPU path)\n", gpu); return 1; }
  CK(xvb_device_check(), "device check");
  {
    char magic[8] = {0};
    FILE* mf = fopen(pos[0], "rb");
    if (!mf || fread(magic, 1, 8, mf) != 8) { fprintf(stderr, "ERROR: xvb-extract: cannot read model file '%s'\n", pos[0]); return 1; }
    fclose(mf);
    if (memcmp(magic, "XVBE0001", 8) == 0) {
      if (ragged) { fprintf(stderr, "ERROR: xvb-extract: --ragged needs a TDNN x-vector model; ECAPA-TDNN has no ragged path yet (drop --ragged)\n"); return 1; }
      CK(xvb_ecapa_load(&r.ec, pos[0]), "loading the ECAPA model");
      r.F = xvb_ecapa_feat_dim(r.ec);
      r.D = xvb_ecapa_embed_dim(r.ec);
    } else {
      CK(xvb_extractor_load(&r.ex, pos[0]), "loading the model");
      r.F = xvb_extractor_feat_dim(pos[0]);
      r.D = xvb_extractor_embed_dim(r.ex);
    }
  }
  xvb_ark_reader_t* in = nullptr;
  FILE* wav_scp = nullptr;
  xvb_fbank_t* fb = nullptr;
  int wav_rate = 0;
  std::vector<float> wave, wav_feats;
  std::string wav_key;
  float* d_wave = nullptr;
  int64_t* d_soff = nullptr;
  size_t wave_cap = 0;
  if (wav_type.empty()) CK(xvb_ark_reader_open(&in, pos[1]), "opening the feature rspecifier");
  else {
    wav_scp = fopen(pos[1], "r");
    if (!wav_scp) { fprintf(stderr, "ERROR: xvb-extract: cannot open wav.scp '%s'\n", pos[1]); return 1; }
    CU(cudaMalloc(&d_soff, 2 * sizeof(int64_t)));
  }
  // next utterance as a host (rows, cols) fp32 matrix: from the ark stream, or wav -> GPU fbank/MFCC
  auto next_utt = [&](const char** key, int* rows, int* cols, const float** data) -> int {
    if (wav_type.empty()) return xvb_ark_reader_next(in, key, rows, cols, data);
    char line[8192];
    for (;;) {
      if (!fgets(line, sizeof line, wav_scp)) return 0;
      char k[4096], path[4096];
      if (sscanf(line, "%4095s %4095[^\n]", k, path) != 2) continue;
      size_t pl = strlen(path);
      while (pl && (path[pl - 1] == ' ' || path[pl - 1] == '\r')) path[--pl] = 0;
      wav_key = k;
      int rate = 0;
      if (!read_wav(path, &wave, &rate)) exit(1);
      if (!fb) {
        wav_rate = rate;
        fo.sample_frequency = (float)rate;
        CK(xvb_fbank_create(&fb, &fo), "xvb_fbank_create");
        if (xvb_fbank_dim(fb) != r.F) { fprintf(stderr, "ERROR: xvb-extract: the feature options give %d dims, the model expects %d\n", xvb_fbank_dim(fb), r.F); exit(1); }
      } else if (rate != wav_rate) { fprintf(stderr, "ERROR: xvb-extract: %s is sampled at %d Hz, the first file at %d Hz\n", k, rate, wav_rate); exit(1); }
      const int64_t n = (int64_t)wave.size(), frames = xvb_fbank_num_frames(fb, n);
      if (frames < 1) { fprintf(stderr, "ERROR: xvb-extract: %s is shorter than one analysis window\n", k); exit(1); }
      if ((size_t)n > wave_cap) { if (d_wave) cudaFree(d_wave); wave_cap = (size_t)n + (size_t)n / 4; CU(cudaMalloc(&d_wave, wave_cap * sizeof(float))); }
      r.reserve((size_t)frames);
      const int64_t soff[2] = {0, n};
      const int32_t foff[2] = {0, (int32_t)frames};
      CU(cudaMemcpy(d_wave, wave.data(), (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
      CU(cudaMemcpy(d_soff, soff, sizeof soff, cudaMemcpyHostToDevice));
      CU(cudaMemcpy(r.d_off, foff, sizeof foff, cudaMemcpyHostToDevice));
      CK(xvb_fbank_compute(fb, d_wave, d_soff, r.d_off, 1, frames, r.d_feats, nullptr), "xvb_fbank_compute");
      wav_feats.resize((size_t)frames * r.F);
      CU(cudaMemcpy(wav_feats.data(), r.d_feats, wav_feats.size() * sizeof(float), cudaMemcpyDeviceToHost));
      *key = wav_key.c_str(); *rows = (int)frames; *cols = r.F; *data = wav_feats.data();
      return 1;
    }
  };
  CK(xvb_ark_writer_open(&r.out, pos[2]), "opening the vector wspecifier");
  CU(cudaMalloc(&r.d_emb, (size_t)r.batch * r.D * sizeof(float)));
  CU(cudaMallocHost(&r.h_emb, (size_t)r.batch * r.D * sizeof(float)));
  CU(cudaMalloc(&r.d_off, ((size_t)r.batch + 2) * sizeof(int32_t)));

  const std::string wspec = pos[2];
  const bool to_stdout = wspec == "-" || (wspec.size() >= 2 && wspec.compare(wspec.size() - 2, 2, ":-") == 0);   // keep the ark stream clean
  std::map<int, std::vector<Item>> buckets;   // frames -> pending chunks of that length
  size_t pending = 0;
  std::vector<Item> window;                   // --ragged: chunks in input order
  size_t window_frames = 0;
  const size_t max_window_frames = 4000000;
  const size_t max_pending = (size_t)r.batch * 64;
  const char* key;
  int rows, cols, rc;
  const float* data;
  std::vector<float> normed;
  while ((rc = next_utt(&key, &rows, &cols, &data)) >= 1) {
    if (rc == 2) { fprintf(stderr, "ERROR: xvb-extract: %s is a double-precision matrix; the extractor takes float32 (FM/CM) features\n", key); return 1; }
    fprintf(to_stdout ? stderr : stdout, "Process utterance for key %s\n", key);   // extract_embeddings.py:81
    if (cols != r.F) { fprintf(stderr, "ERROR: xvb-extract: %s has %d-dim features, the model expects %d\n", key, cols, r.F); return 1; }
    if (rows < 1) { fprintf(stderr, "ERROR: xvb-extract: %s has no frames\n", key); return 1; }
    if (r.cmn) {   // whole utterance, before the chunk rule (the reference normalises upstream of the model)
      r.reserve((size_t)rows);
      CU(cudaMemcpy(r.d_feats, data, (size_t)rows * cols * sizeof(float), cudaMemcpyHostToDevice));
      r.cmn_device(r.d_feats, r.d_tmp, {0, rows});
      normed.resize((size_t)rows * cols);
      CU(cudaMemcpy(normed.data(), r.d_tmp, normed.size() * sizeof(float), cudaMemcpyDeviceToHost));
      data = normed.data();
    }
    Utt u;
    u.key = key;
    u.frames = rows;
    const int num_split = (rows + max_chunk - 1) / max_chunk, split = rows / num_split;
    u.pending = num_split;
    const int ui = (int)r.utts.size();
    r.utts.push_back(u);
    for (int c = 0, off = 0; c < num_split; ++c) {
      const int len = c + 1 < num_split ? split : rows - off;
      Item it;
      it.utt = ui;
      it.frames = len;
      it.feats.assign(data + (size_t)off * cols, data + (size_t)(off + len) * cols);
      off += len;
      if (ragged) {
        window.push_back(std::move(it));
        window_frames += len;
        continue;
      }
      std::vector<Item>& b = buckets[len];
      b.push_back(std::move(it));
      ++pending;
      if ((int)b.size() == r.batch) { pending -= b.size(); r.run(b); }
    }
    if (window_frames >= max_window_frames) {
      r.run_ragged(window);
      window_frames = 0;
    }
    if (pending > max_pending) {   // bound host memory: flush the fullest bucket
      auto best = buckets.begin();
      for (auto it = buckets.begin(); it != buckets.end(); ++it)
        if (it->second.size() > best->second.size()) best = it;
      pending -= best->second.size();
      r.run(best->second);
    }
  }
  if (rc < 0) die("reading features");
  for (auto& kv : buckets) r.run(kv.second);
  r.run_ragged(window);
  if (in) xvb_ark_reader_close(in);
  if (wav_scp) fclose(wav_scp);
  if (fb) xvb_fbank_destroy(fb);
  CK(xvb_ark_writer_close(r.out), "closing the vector wspecifier");
  if (r.ex) xvb_extractor_destroy(r.ex);
  if (r.ec) xvb_ecapa_destroy(r.ec);
  fprintf(stderr, "xvb-extract: %ld utterances, %ld frames\n", r.done_utts, r.done_frames);
  return 0;
}
