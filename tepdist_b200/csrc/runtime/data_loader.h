// Native input pipeline: memory-mapped token files -> (tokens, labels) batches in caller-provided (pinned) host buffers, filled
// by background threads a few steps ahead of the training loop.
//
// Reference parity (SURVEY K13 / F: examples/GPT2/inputs.py): the reference's client reads BPE token records through a
// tf.data pipeline -- windows of n_ctx + 1 tokens cut into (input, next-token label), several datasets mixed by weight
// (sample_from_datasets), prefetch a few batches, and a `fake_input` mode of random tokens.  Here the same capabilities without
// a framework dependency, designed around what the training step needs on a B200 box: batches land directly in page-locked memory
// that the step copies from asynchronously, and sampling is STATELESS -- sample k of the run is a pure function of (seed, k) --
// so every data-parallel rank computes exactly its own rows of every global batch without coordination, and a resumed job
// continues the stream from its step counter alone.
#pragma once
#include <atomic>
#include <condition_variable>
#include <cstdint>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

namespace tepdist {

// One flat binary file of token ids (little-endian uint16 or int32), memory-mapped read-only.
class TokenFile {
 public:
  TokenFile(const std::string& path, int bytes_per_token);
  ~TokenFile();
  TokenFile(const TokenFile&) = delete;
  TokenFile& operator=(const TokenFile&) = delete;
  uint64_t num_tokens() const { return n_tokens_; }
  int32_t at(uint64_t i) const;
  const std::string& path() const { return path_; }

 private:
  std::string path_;
  int fd_ = -1;
  const uint8_t* base_ = nullptr;
  uint64_t bytes_ = 0, n_tokens_ = 0;
  int bpt_ = 2;
};

// A weighted mixture of datasets, each a set of token files; `vocab` > 0 switches to synthetic tokens (the reference's fake_input).
class TokenSource {
 public:
  // files[d] = the files of dataset d, weights[d] its sampling weight (any positive scale)
  void AddDataset(const std::vector<std::string>& files, double weight, int bytes_per_token);
  void SetSynthetic(int vocab) { synthetic_vocab_ = vocab; }
  bool synthetic() const { return synthetic_vocab_ > 0; }
  uint64_t total_tokens() const;
  int num_datasets() const { return (int)datasets_.size(); }
  // Window `sample_id` of the run: n consecutive tokens (n = n_ctx + 1).  Pure function of (seed, sample_id).
  void Sample(uint64_t seed, uint64_t sample_id, int n, int32_t* out) const;
  // which dataset / file / offset `sample_id` maps to (tests, debugging)
  void Locate(uint64_t seed, uint64_t sample_id, int n, int* dataset, int* file, uint64_t* offset) const;

 private:
  struct Dataset {
    std::vector<std::unique_ptr<TokenFile>> files;
    double weight = 1.0;
  };
  std::vector<Dataset> datasets_;
  int synthetic_vocab_ = 0;
};

// Fills a ring of host buffers with this rank's rows of consecutive global batches.
//   global batch t = samples [t * global_batch, (t + 1) * global_batch); rank r takes rows [r * batch, (r + 1) * batch) of it.
class BatchLoader {
 public:
  BatchLoader(std::shared_ptr<TokenSource> src, int batch, int n_ctx, int rank, int world, uint64_t seed, int threads);
  ~BatchLoader();
  // slot buffers: int32 [batch, n_ctx] each, owned by the caller (torch pinned tensors) and alive until Stop().
  // Optional `segments` buffers (one per slot, or none) receive document ids: seg[i] = number of `eot` tokens at window
  // positions < i, so the end-of-text token belongs to the document it ends.
  void SetBuffers(const std::vector<uintptr_t>& tokens, const std::vector<uintptr_t>& labels,
                  const std::vector<uintptr_t>& segments = {}, int32_t eot = 0);
  void Start(uint64_t first_step);
  // Blocks until the batch of the next step is complete; returns its slot.  Steps are handed out in order.
  int Acquire(uint64_t* step);
  void Release(int slot);
  void Stop();
  int num_slots() const { return (int)tok_.size(); }
  uint64_t batches_filled() const { return filled_.load(); }

 private:
  void Worker();
  void Fill(int slot, uint64_t step);

  std::shared_ptr<TokenSource> src_;
  int batch_, n_ctx_, rank_, world_, threads_;
  uint64_t seed_;
  std::vector<int32_t*> tok_, lab_, seg_;
  int32_t eot_ = 0;
  // slot state machine: kFree -> (claimed by a worker for step s) kFilling -> kReady -> (Acquire) kInUse -> (Release) kFree
  enum State { kFree, kFilling, kReady, kInUse };
  std::vector<State> state_;
  std::vector<uint64_t> slot_step_;
  uint64_t next_fill_ = 0, next_out_ = 0;
  std::mutex mu_;
  std::condition_variable cv_;
  std::vector<std::thread> workers_;
  bool running_ = false, stop_ = false;
  std::string error_;        // first exception of a worker thread; re-raised by Acquire
  std::atomic<uint64_t> filled_{0};
};

}  // namespace tepdist
