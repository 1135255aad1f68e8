#include "runtime/data_loader.h"

#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <cstring>
#include <memory>
#include <stdexcept>

namespace tepdist {

namespace {
// splitmix64: a full-period 64-bit mixer; stream position -> value is a pure function (no generator state to carry around)
inline uint64_t Mix(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
inline uint64_t Draw(uint64_t seed, uint64_t sample, uint64_t lane) { return Mix(Mix(seed ^ 0xD1B54A32D192ED03ull) + Mix(sample) * 3 + lane); }
inline double Unit(uint64_t r) { return (double)(r >> 11) * (1.0 / 9007199254740992.0); }   // [0, 1)
}  // namespace

// ------------------------------------------------------------------------------------------------ TokenFile
TokenFile::TokenFile(const std::string& path, int bytes_per_token) : path_(path), bpt_(bytes_per_token) {
  if (bpt_ != 2 && bpt_ != 4) throw std::invalid_argument("token files hold uint16 or int32 ids (bytes_per_token 2 or 4)");
  fd_ = ::open(path.c_str(), O_RDONLY);
  if (fd_ < 0) throw std::runtime_error("cannot open token file " + path);
  struct stat st;
  if (::fstat(fd_, &st) != 0 || st.st_size <= 0) {
    ::close(fd_);
    throw std::runtime_error("empty or unreadable token file " + path);
  }
  bytes_ = (uint64_t)st.st_size;
  n_tokens_ = bytes_ / (uint64_t)bpt_;
  void* p = ::mmap(nullptr, bytes_, PROT_READ, MAP_SHARED, fd_, 0);
  if (p == MAP_FAILED) {
    ::close(fd_);
    throw std::runtime_error("mmap failed for " + path);
  }
  base_ = (const uint8_t*)p;
  ::madvise(p, bytes_, MADV_RANDOM);   // windows are drawn at random offsets: no read-ahead beyond the window
}
TokenFile::~TokenFile() {
  if (base_) ::munmap((void*)base_, bytes_);
  if (fd_ >= 0) ::close(fd_);
}
int32_t TokenFile::at(uint64_t i) const {
  if (bpt_ == 2) {
    uint16_t v;
    std::memcpy(&v, base_ + 2 * i, 2);
    return (int32_t)v;
  }
  int32_t v;
  std::memcpy(&v, base_ + 4 * i, 4);
  return v;
}

// ------------------------------------------------------------------------------------------------ TokenSource
void TokenSource::AddDataset(const std::vector<std::string>& files, double weight, int bytes_per_token) {
  if (files.empty() || !(weight > 0)) throw std::invalid_argument("a dataset needs at least one file and a positive weight");
  Dataset d;
  d.weight = weight;
  for (auto& f : files) d.files.push_back(std::make_unique<TokenFile>(f, bytes_per_token));
  datasets_.push_back(std::move(d));
}
uint64_t TokenSource::total_tokens() const {
  uint64_t t = 0;
  for (auto& d : datasets_)
    for (auto& f : d.files) t += f->num_tokens();
  return t;
}
void TokenSource::Locate(uint64_t seed, uint64_t sample_id, int n, int* dataset, int* file, uint64_t* offset) const {
  if (datasets_.empty()) throw std::runtime_error("no dataset");
  // dataset by weight
  double total = 0;
  for (auto& d : datasets_) total += d.weight;
  double u = Unit(Draw(seed, sample_id, 0)) * total;
  int di = 0;
  for (; di + 1 < (int)datasets_.size(); ++di) {
    if (u < datasets_[di].weight) break;
    u -= datasets_[di].weight;
  }
  const Dataset& d = datasets_[di];
  // window uniformly over every valid start position of every file of the dataset (longer files get proportionally more draws)
  uint64_t windows = 0;
  std::vector<uint64_t> per(d.files.size());
  for (size_t i = 0; i < d.files.size(); ++i) {
    per[i] = d.files[i]->num_tokens() >= (uint64_t)n ? d.files[i]->num_tokens() - (uint64_t)n + 1 : 0;
    windows += per[i];
  }
  if (windows == 0) throw std::runtime_error("every file of dataset " + std::to_string(di) + " is shorter than one window");
  uint64_t w = Draw(seed, sample_id, 1) % windows;
  size_t fi = 0;
  while (w >= per[fi]) w -= per[fi++];
  *dataset = di;
  *file = (int)fi;
  *offset = w;
}
void TokenSource::Sample(uint64_t seed, uint64_t sample_id, int n, int32_t* out) const {
  if (synthetic()) {
    for (int i = 0; i < n; ++i) out[i] = (int32_t)(Draw(seed, sample_id, 2 + (uint64_t)i) % (uint64_t)synthetic_vocab_);
    return;
  }
  int di, fi;
  uint64_t off;
  Locate(seed, sample_id, n, &di, &fi, &off);
  const TokenFile& f = *datasets_[di].files[fi];
  for (int i = 0; i < n; ++i) out[i] = f.at(off + (uint64_t)i);
}

// ------------------------------------------------------------------------------------------------ BatchLoader
BatchLoader::BatchLoader(std::shared_ptr<TokenSource> src, int batch, int n_ctx, int rank, int world, uint64_t seed, int threads)
    : src_(std::move(src)), batch_(batch), n_ctx_(n_ctx), rank_(rank), world_(world), threads_(std::max(1, threads)), seed_(seed) {
  if (batch <= 0 || n_ctx <= 0 || world <= 0 || rank < 0 || rank >= world) throw std::invalid_argument("bad loader geometry");
}
BatchLoader::~BatchLoader() { Stop(); }

void BatchLoader::SetBuffers(const std::vector<uintptr_t>& tokens, const std::vector<uintptr_t>& labels,
                             const std::vector<uintptr_t>& segments, int32_t eot) {
  if (running_) throw std::runtime_error("SetBuffers while running");
  if (tokens.empty() || tokens.size() != labels.size()) throw std::invalid_argument("need one tokens and one labels buffer per slot");
  if (!segments.empty() && segments.size() != tokens.size()) throw std::invalid_argument("need one segments buffer per slot, or none");
  tok_.clear();
  lab_.clear();
  seg_.clear();
  for (auto p : tokens) tok_.push_back(reinterpret_cast<int32_t*>(p));
  for (auto p : labels) lab_.push_back(reinterpret_cast<int32_t*>(p));
  for (auto p : segments) seg_.push_back(reinterpret_cast<int32_t*>(p));
  eot_ = eot;
  state_.assign(tok_.size(), kFree);
  slot_step_.assign(tok_.size(), 0);
}

void BatchLoader::Start(uint64_t first_step) {
  if (running_) throw std::runtime_error("loader already running");
  if (tok_.empty()) throw std::runtime_error("SetBuffers first");
  next_fill_ = next_out_ = first_step;
  std::fill(state_.begin(), state_.end(), kFree);
  stop_ = false;
  error_.clear();
  running_ = true;
  for (int i = 0; i < threads_; ++i) workers_.emplace_back(&BatchLoader::Worker, this);
}

void BatchLoader::Stop() {
  {
    std::lock_guard<std::mutex> l(mu_);
    if (!running_) return;
    stop_ = true;
  }
  cv_.notify_all();
  for (auto& t : workers_) t.join();
  workers_.clear();
  running_ = false;
}

void BatchLoader::Fill(int slot, uint64_t step) {
  const int n = n_ctx_ + 1;
  std::vector<int32_t> win((size_t)n);
  const uint64_t global_batch = (uint64_t)batch_ * (uint64_t)world_;
  for (int b = 0; b < batch_; ++b) {
    const uint64_t sample = step * global_batch + (uint64_t)rank_ * (uint64_t)batch_ + (uint64_t)b;
    src_->Sample(seed_, sample, n, win.data());
    std::memcpy(tok_[slot] + (size_t)b * n_ctx_, win.data(), sizeof(int32_t) * (size_t)n_ctx_);
    std::memcpy(lab_[slot] + (size_t)b * n_ctx_, win.data() + 1, sizeof(int32_t) * (size_t)n_ctx_);   // next-token labels
    if (!seg_.empty()) {
      int32_t* seg = seg_[slot] + (size_t)b * n_ctx_;
      int32_t d = 0;
      for (int i = 0; i < n_ctx_; ++i) {
        seg[i] = d;
        d += win[(size_t)i] == eot_;
      }
    }
  }
}

void BatchLoader::Worker() {
  const int S = (int)tok_.size();
  for (;;) {
    uint64_t step;
    int slot;
    {
      std::unique_lock<std::mutex> l(mu_);
      cv_.wait(l, [&] { return stop_ || state_[next_fill_ % S] == kFree; });
      if (stop_) return;
      step = next_fill_++;
      slot = (int)(step % S);
      state_[slot] = kFilling;
      slot_step_[slot] = step;
    }
    try {
      Fill(slot, step);
    } catch (const std::exception& e) {
      // (a worker thread must not let an exception escape: it is handed to the consumer, which re-raises it from Acquire)
      {
        std::lock_guard<std::mutex> l(mu_);
        if (error_.empty()) error_ = e.what();
        stop_ = true;
      }
      cv_.notify_all();
      return;
    }
    {
      std::lock_guard<std::mutex> l(mu_);
      state_[slot] = kReady;
      ++filled_;
    }
    cv_.notify_all();
  }
}

int BatchLoader::Acquire(uint64_t* step) {
  const int S = (int)tok_.size();
  std::unique_lock<std::mutex> l(mu_);
  if (!running_) throw std::runtime_error("loader not running");
  const int slot = (int)(next_out_ % S);
  cv_.wait(l, [&] { return stop_ || (state_[slot] == kReady && slot_step_[slot] == next_out_); });
  if (stop_) throw std::runtime_error(error_.empty() ? std::string("loader stopped") : "data loader: " + error_);
  state_[slot] = kInUse;
  if (step) *step = next_out_;
  ++next_out_;
  return slot;
}

void BatchLoader::Release(int slot) {
  {
    std::lock_guard<std::mutex> l(mu_);
    if (slot < 0 || slot >= (int)state_.size() || state_[slot] != kInUse) throw std::runtime_error("Release of a slot that is not in use");
    state_[slot] = kFree;
  }
  cv_.notify_all();
}

}  // namespace tepdist
