// libbmbs_gpu.so: C ABI (include/bmbs.h) over the kernels in bmbs_kernels.cuh.
// Index files are read exactly as the reference writes them (bwt.cpp:1704-1835, :2080-2084; Index.cpp:134-159,
// :827-828) and re-laid out for the GPU at load time; nothing is written back.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <vector>
#include "bmbs_kernels.cuh"

using namespace bmbs;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& m) { g_err = m; return code; }

#define CU(call) do { cudaError_t e_ = (call); if (e_ != cudaSuccess) return fail(BMBS_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); } while (0)

// splits [0, n) over a few host threads (index re-layout at load)
template <class F> void parallel_for(u64 n, F fn) {
  unsigned hw = std::thread::hardware_concurrency();
  const u64 T = std::max<u64>(1, std::min<u64>(hw ? hw : 4, 16));
  std::vector<std::thread> th;
  for (u64 t = 1; t < T; ++t) th.emplace_back([=] { fn(n * t / T, n * (t + 1) / T); });
  fn(0, n / T);
  for (auto& x : th) x.join();
}

// The index files are mapped, not read: the arrays go from the page cache straight to the device, where they are
// re-laid out (DESIGN.md 3); nothing is copied or converted on the host.
struct MappedFile {
  char* p = nullptr; size_t size = 0;
  bool open(const std::string& path) {
    const int fd = ::open(path.c_str(), O_RDONLY);
    if (fd < 0) return false;
    struct stat st;
    if (fstat(fd, &st) != 0 || st.st_size <= 0) { ::close(fd); return false; }
    void* m = mmap(nullptr, (size_t)st.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
    ::close(fd);
    if (m == MAP_FAILED) return false;
    p = (char*)m; size = (size_t)st.st_size;
    madvise(p, size, MADV_WILLNEED);
    return true;
  }
  ~MappedFile() { if (p) munmap(p, size); }
};
template <class T> struct Span { const T* p = nullptr; size_t n = 0; size_t bytes() const { return n * sizeof(T); } };

struct HostIndex {
  u64 sa_length = 0, shapline = 0, nacgt[5] = {0, 0, 0, 0, 0}, N = 0;
  MappedFile f_pac, f_bwt, f_sa, f_occ;
  Span<u64> bwt, high_occ, sa_flag;
  Span<u32> hash_hi, ssa;
  Span<uint8_t> hash_lo, pac;
  std::vector<u64> chrom_start;      // chrom_start[i] = first coordinate of chromosome i, one more entry = N
};

// u64 count followed by `count` elements at `off`; advances off
template <class T> bool take(const MappedFile& f, size_t& off, Span<T>& out) {
  if (off + 8 > f.size) return false;
  u64 n; memcpy(&n, f.p + off, 8); off += 8;
  if (n > (f.size - off) / sizeof(T)) return false;
  out.p = (const T*)(f.p + off); out.n = (size_t)n; off += (size_t)n * sizeof(T);
  return true;
}

int load_files(const std::string& prefix, HostIndex& h) {
  FILE* f = fopen(prefix.c_str(), "rb");
  if (!f) return fail(BMBS_ERR_IO, "cannot open " + prefix);
  u64 nc = 0; bool ok = fread(&nc, 8, 1, f) == 1;
  u64 at = 0;
  for (u64 i = 0; ok && i < nc; ++i) { u64 l = 0, cl = 0; ok = fread(&l, 8, 1, f) == 1 && fseek(f, (long)l, SEEK_CUR) == 0 && fread(&cl, 8, 1, f) == 1; h.chrom_start.push_back(at); at += cl; }
  ok = ok && fread(&h.N, 8, 1, f) == 1; fclose(f);
  h.chrom_start.push_back(at);
  if (!ok) return fail(BMBS_ERR_IO, "short read in " + prefix);
  if (!h.f_pac.open(prefix + ".bs.pac")) return fail(BMBS_ERR_IO, "cannot open " + prefix + ".bs.pac");
  size_t off = 0;
  if (!take(h.f_pac, off, h.pac) || h.pac.n < (h.N + 3) / 4) return fail(BMBS_ERR_IO, "short read in " + prefix + ".bs.pac");
  const std::string p = prefix + ".bs.index";
  f = fopen(p.c_str(), "rb");
  if (!f) return fail(BMBS_ERR_IO, "cannot open " + p);
  ok = fread(&h.sa_length, 8, 1, f) == 1 && fread(&h.shapline, 8, 1, f) == 1 && fread(h.nacgt, 8, 5, f) == 5; fclose(f);
  if (!ok) return fail(BMBS_ERR_IO, "short read in " + p);
  if (!h.f_bwt.open(p + ".bwt")) return fail(BMBS_ERR_IO, "cannot open " + p + ".bwt");
  off = 0;
  if (!take(h.f_bwt, off, h.bwt)) return fail(BMBS_ERR_IO, "short read in " + p + ".bwt");
  {   // u64 n; u32 hi[n]; u8 lo[n]
    if (off + 8 > h.f_bwt.size) return fail(BMBS_ERR_IO, "short read in " + p + ".bwt");
    u64 n; memcpy(&n, h.f_bwt.p + off, 8); off += 8;
    if (n > (h.f_bwt.size - off) / 5) return fail(BMBS_ERR_IO, "short read in " + p + ".bwt");
    h.hash_hi.p = (const u32*)(h.f_bwt.p + off); h.hash_hi.n = (size_t)n; off += (size_t)n * 4;
    h.hash_lo.p = (const uint8_t*)(h.f_bwt.p + off); h.hash_lo.n = (size_t)n;
  }
  if (!h.f_sa.open(p + ".sa")) return fail(BMBS_ERR_IO, "cannot open " + p + ".sa");
  off = 0;
  if (!take(h.f_sa, off, h.ssa) || !take(h.f_sa, off, h.sa_flag)) return fail(BMBS_ERR_IO, "short read in " + p + ".sa");
  if (!h.f_occ.open(p + ".occ")) return fail(BMBS_ERR_IO, "cannot open " + p + ".occ");
  off = 0;
  if (!take(h.f_occ, off, h.high_occ)) return fail(BMBS_ERR_IO, "short read in " + p + ".occ");
  if (h.sa_length != 2 * h.N + 1) return fail(BMBS_ERR_IO, "index header does not match the genome length");
  // fault the mappings in with a few threads (the driver's pageable copy would otherwise take the page faults one by one)
  const MappedFile* files[4] = {&h.f_pac, &h.f_bwt, &h.f_sa, &h.f_occ};
  for (const MappedFile* mf : files) {
    const size_t pages = (mf->size + 4095) / 4096;
    std::atomic<unsigned> sink(0);
    parallel_for(pages, [&](u64 lo, u64 hi) { unsigned x = 0; for (u64 i = lo; i < hi; ++i) x += (unsigned char)mf->p[i * 4096]; sink += x; });
  }
  return BMBS_OK;
}

struct DeviceCopy {
  int dev = 0; DevIndex view{}; size_t bytes = 0;
  int grid_sms = 148;        // SMs the persistent and grid-stride launches of batches and refiners are sized for (BMBS_GRID_SMS)
  void *occ = nullptr, *flag = nullptr, *hash = nullptr, *ssa = nullptr, *planes = nullptr, *dsa_lo = nullptr, *dsa_hi = nullptr, *ktab = nullptr, *chroms = nullptr;
};

// ---- deep seed table (kmer_entry, bmbs_device.cuh): one thread per 16-mer walks the <= 3^D extensions depth first, sharing
// the LF steps of common prefixes and stopping where the reference's greedy loop would stop
__device__ __forceinline__ void ktab_fill(u64* t, u32 first, u32 stride, u32 count, u64 e) {
  for (u32 i = 0; i < count; ++i) t[first + i * stride] = e;
}
template <int LEFT>
__device__ void ktab_node(const DevIndex& ix, u64* t, u32 prefix, u32 stride, u32 m, u64 top, u64 bot) {
  // node: symbols 16..m-1 fixed (extension value `prefix`, next digit weighs `stride`), interval [top, bot) not empty
  constexpr u32 below = LEFT == 0 ? 1 : LEFT == 1 ? 3 : LEFT == 2 ? 9 : LEFT == 3 ? 27 : 81;
  if (bot - top == 1) { int st; const u64 sa = locate_row(ix, top, st); ktab_fill(t, prefix, stride, below, kmer_entry(m, sa, sa + 1)); return; }   // one row: store its SA value
  if (LEFT == 0) { ktab_fill(t, prefix, stride, below, kmer_entry(m, top, bot)); return; }
  if constexpr (LEFT > 0) {
    for (int c = 0; c < 3; ++c) {
      u64 a = top, b = bot;
      lf_pair(ix, a, b, c);
      if (b <= a) ktab_fill(t, prefix + c * stride, stride * 3, below / 3, kmer_entry(m, top, bot));
      else ktab_node<LEFT - 1>(ix, t, prefix + c * stride, stride * 3, m + 1, a, b);
    }
  }
}
template <int D>
__global__ void __launch_bounds__(128) build_ktab(DevIndex ix, u64* table, u32 n_keys) {
  constexpr u32 leaves = D == 1 ? 3 : D == 2 ? 9 : D == 3 ? 27 : 81;
  for (u32 key = blockIdx.x * blockDim.x + threadIdx.x; key < n_keys; key += gridDim.x * blockDim.x) {
    u64* t = table + (u64)key * leaves;
    u64 top, bot; hash_query(ix, key, top, bot);
    if (bot <= top) ktab_fill(t, 0, 1, leaves, 0ull);
    else ktab_node<D>(ix, t, 0, 1, 16, top, bot);
  }
}

// ---- re-layout of the on-disk arrays, on the device (formats: SURVEY.md 8a D1-D7)
// occ blocks: fold the 65536-row table and the 16-bit counters of the 40-byte superblocks (bwt.h:1007-1058) into absolute counts
__global__ void relayout_occ(const u64* __restrict__ bwt, u64 bwt_words, const u64* __restrict__ high_occ, u64 high_words, u64 nblk, u64* __restrict__ occ) {
  for (u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x; b < nblk; b += (u64)gridDim.x * blockDim.x) {
    const u64 sb = (b >> 1) * 5, sub = b & 1, w = sb + 1 + 2 * sub, hi_i = ((b << 6) >> 16) * 2;
    u64 o0 = 0, o1 = 0, o2 = 0, o3 = 0;
    if (w + 1 < bwt_words && hi_i + 1 < high_words) {
      const u64 hdr = bwt[sb];
      o0 = bwt[w]; o1 = bwt[w + 1];
      o2 = high_occ[hi_i] + ((hdr >> (48 - 32 * sub)) & 0xFFFF);
      o3 = high_occ[hi_i + 1] + ((hdr >> (32 - 32 * sub)) & 0xFFFF);
    }
    occ[b * 4] = o0; occ[b * 4 + 1] = o1; occ[b * 4 + 2] = o2; occ[b * 4 + 3] = o3;
  }
}
// flag blocks of 64 rows with the rank of the block start (reference: 5 words per 256 rows, bwt.h:2449-2560).  The flag file's
// last word is uninitialised in reference-built indexes (bwt.cpp:1188-1192 vs :1657-1664): bits beyond the last row are masked.
__global__ void relayout_flag(const u64* __restrict__ sa_flag, u64 flag_words, u64 nfb, u64 last_row, u64* __restrict__ flag) {
  for (u64 b = (u64)blockIdx.x * blockDim.x + threadIdx.x; b < nfb; b += (u64)gridDim.x * blockDim.x) {
    const u64 g = (b >> 2) * 5, in = b & 3;
    u64 bits = 0, rank = 0;
    if (g + 1 + in < flag_words) {
      rank = sa_flag[g];
      for (u64 t = 0; t < in; ++t) rank += (u64)__popcll(sa_flag[g + 1 + t]);
      bits = sa_flag[g + 1 + in];
    }
    const u64 lb = last_row >> 6, used = (last_row & 63) + 1;
    if (b == lb && used < 64) bits &= ~0ull << (64 - used);
    if (b > lb) bits = 0;
    flag[b * 2] = bits; flag[b * 2 + 1] = rank;
  }
}
// 16-mer table: u32 + u8 per entry (bwt.h:284-306) -> one u64
__global__ void relayout_hash(const u32* __restrict__ hi, const unsigned char* __restrict__ lo, u64 n, u64* __restrict__ hash) {
  for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
    hash[i] = ((u64)(hi[i] & 0x0FFFFFFFu) << 8) | lo[i] | ((u64)(hi[i] >> 28) << 60);
}
// bit-planes of G ++ revcomp(G) from the 2-bit genome (Index.cpp:734-831: four bases per byte, first base in the top bits)
__global__ void relayout_planes(const unsigned char* __restrict__ pac, u64 N, u64 n_words, uint2* __restrict__ planes) {
  const u64 n = 2 * N;
  for (u64 w = (u64)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (u64)gridDim.x * blockDim.x) {
    u32 x = 0, y = 0;
    for (u32 t = 0; t < 32; ++t) {
      const u64 pos = w * 32 + t;
      if (pos >= n) break;
      u32 c;
      if (pos < N) c = (pac[pos >> 2] >> (6 - 2 * (pos & 3))) & 3;
      else { const u64 i = n - 1 - pos; c = 3 - ((pac[i >> 2] >> (6 - 2 * (i & 3))) & 3); }
      x |= (c & 1u) << t; y |= (c >> 1) << t;
    }
    planes[w] = make_uint2(x, y);
  }
}

// every row's suffix-array value from the sampled one, once per index load (the same walk the reference does per hit)
__global__ void __launch_bounds__(256) densify_sa(DevIndex ix, u32* lo, unsigned char* hi) {
  for (u64 row = (u64)blockIdx.x * blockDim.x + threadIdx.x; row < ix.n_rows; row += (u64)gridDim.x * blockDim.x) {
    int st; const u64 sa = locate_row_walk(ix, row, st);
    lo[row] = (u32)sa;
    if (hi) hi[row] = (unsigned char)(sa >> 32);
  }
}

}  // namespace

// every loaded index gets a serial that is never reused: the one-call forms cache their batch contexts per thread and
// must not mistake a new index that malloc placed at a freed handle's address for the old one
namespace {
std::mutex g_live_mu; std::set<u64> g_live_serials; std::atomic<u64> g_next_serial{1};
bool serial_live(u64 s) { std::lock_guard<std::mutex> l(g_live_mu); return g_live_serials.count(s) != 0; }
}  // namespace

struct bmbs_index {
  u64 N = 0;
  u64 serial = 0;
  std::vector<DeviceCopy> copies;
  const DeviceCopy* on(int dev) const { for (auto& c : copies) if (c.dev == dev) return &c; return nullptr; }
};

extern "C" const char* bmbs_last_error(void) { return g_err.c_str(); }
extern "C" void bmbs_params_default(bmbs_params* p) { p->e_rate = 0.08; p->seed_len = 30; p->min_ins = 0; p->max_ins = 500; p->sensitive = 0; p->ambiguous_out = 0; }
extern "C" uint64_t bmbs_index_genome_length(const bmbs_index* idx) { return idx ? idx->N : 0; }
extern "C" uint64_t bmbs_index_device_bytes(const bmbs_index* idx) { return idx && !idx->copies.empty() ? idx->copies[0].bytes : 0; }

extern "C" void bmbs_index_free(bmbs_index* idx) {
  if (!idx) return;
  { std::lock_guard<std::mutex> l(g_live_mu); g_live_serials.erase(idx->serial); }
  for (auto& c : idx->copies) { cudaSetDevice(c.dev); cudaFree(c.occ); cudaFree(c.flag); cudaFree(c.hash); cudaFree(c.ssa); cudaFree(c.planes); cudaFree(c.dsa_lo); cudaFree(c.dsa_hi); cudaFree(c.ktab); cudaFree(c.chroms); }
  delete idx;
}

extern "C" int bmbs_index_load(const char* index_prefix, const int* devices, int n_dev, bmbs_index** out) {
  if (!index_prefix || !out) return fail(BMBS_ERR_ARG, "null argument");
  HostIndex h;
  const bool verbose = getenv("BMBS_VERBOSE") != nullptr;
  auto tnow = [] { timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return ts.tv_sec + ts.tv_nsec * 1e-9; };
  double t_prev = tnow();
  auto lap = [&](const char* what) { if (verbose) { const double t = tnow(); fprintf(stderr, "[bmbs load] %-28s %.3f s\n", what, t - t_prev); t_prev = t; } };
  // CUDA context creation overlaps the file reads and the host re-layout
  int dev0 = 0;
  if (!devices || n_dev <= 0) { devices = &dev0; n_dev = 1; }
  // CUDA contexts are created while the files are mapped, one thread per device
  std::vector<std::thread> warm;
  // (host threads that wait for the device sleep instead of spinning -- the mapper runs more threads than cores; BMBS_SPIN=1 keeps
  // the driver's default.  No effect when the process already has a context on the device.)
  const bool spin = getenv("BMBS_SPIN") != nullptr;
  for (int d = 0; d < n_dev; ++d) warm.emplace_back([=] { cudaSetDevice(devices[d]); if (!spin) { cudaSetDeviceFlags(cudaDeviceScheduleBlockingSync); cudaGetLastError(); } cudaFree(0); });
  auto warm_join = [&] { for (auto& t : warm) t.join(); };
  int rc = load_files(index_prefix, h);
  if (rc) { warm_join(); return rc; }
  lap("map index files");
  const u64 n = 2 * h.N;                       // text length = BWT symbols
  const u64 nblk = (n >> 6) + 2, nfb = (h.sa_length >> 6) + 2, npw = (n + 31) / 32 + 64;
  const size_t nh = h.hash_hi.n;

  bmbs_index* idx = new bmbs_index();
  idx->N = h.N;
  idx->serial = g_next_serial++;
  { std::lock_guard<std::mutex> l(g_live_mu); g_live_serials.insert(idx->serial); }
  warm_join();
  lap("(wait for the CUDA context)");
  // every device uploads the raw arrays over its own link and builds its layouts itself: one host thread per device
  // (the loads of an 8-GPU run overlap instead of queueing behind each other)
  idx->copies.resize((size_t)n_dev);
  std::vector<std::string> errors((size_t)n_dev);
  auto load_on = [&](int d) {
    std::string& err_out = errors[(size_t)d];
    DeviceCopy& c = idx->copies[(size_t)d]; c.dev = devices[d];
    const bool lap_here = d == 0;
    auto lap = [&](const char* what) { if (verbose && lap_here) { const double t = tnow(); fprintf(stderr, "[bmbs load] %-28s %.3f s\n", what, t - t_prev); t_prev = t; } };
    cudaError_t e = cudaSetDevice(c.dev);
    cudaDeviceProp prop; if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, c.dev);
    const int grid = e == cudaSuccess ? prop.multiProcessorCount * 16 : 1;
    // BMBS_GRID_SMS=n sizes the persistent and grid-stride launches of every batch and refiner on this copy for min(n, SMs) SMs
    // (tests: a batch of a few thousand reads then gives each lane, warp and block of those kernels many items in turn, so
    // the reset of per-item state between items runs everywhere)
    if (e == cudaSuccess) {
      c.grid_sms = prop.multiProcessorCount;
      if (const char* gs = getenv("BMBS_GRID_SMS")) { const int g = atoi(gs); if (g >= 1) c.grid_sms = std::min(g, c.grid_sms); }
    }
    // raw file arrays -> device (16 zero words of slack behind bwt and sa_flag, as the re-layout reads a little past the end)
    void *r_bwt = nullptr, *r_high = nullptr, *r_flag = nullptr, *r_hi = nullptr, *r_lo = nullptr, *r_pac = nullptr;
    auto raw = [&](void** p, const void* src, size_t bytes, size_t slack) -> cudaError_t {
      cudaError_t x = cudaMalloc(p, bytes + slack + 16); if (x != cudaSuccess) return x;
      if (slack) { x = cudaMemset((char*)*p + bytes, 0, slack); if (x != cudaSuccess) return x; }
      return bytes ? cudaMemcpy(*p, src, bytes, cudaMemcpyHostToDevice) : cudaSuccess;
    };
    auto dev_alloc = [&](void** p, size_t bytes) -> cudaError_t { c.bytes += bytes; return cudaMalloc(p, bytes); };
    if (e == cudaSuccess) e = raw(&r_bwt, h.bwt.p, h.bwt.bytes(), 128);
    if (e == cudaSuccess) e = raw(&r_high, h.high_occ.p, h.high_occ.bytes(), 0);
    if (e == cudaSuccess) e = dev_alloc(&c.occ, nblk * 32);
    if (e == cudaSuccess) { relayout_occ<<<grid, 256>>>((const u64*)r_bwt, h.bwt.n + 16, (const u64*)r_high, h.high_occ.n, nblk, (u64*)c.occ); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = raw(&r_flag, h.sa_flag.p, h.sa_flag.bytes(), 128);
    if (e == cudaSuccess) e = dev_alloc(&c.flag, nfb * 16);
    if (e == cudaSuccess) { relayout_flag<<<grid, 256>>>((const u64*)r_flag, h.sa_flag.n + 16, nfb, h.sa_length - 1, (u64*)c.flag); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = raw(&r_hi, h.hash_hi.p, h.hash_hi.bytes(), 0);
    if (e == cudaSuccess) e = raw(&r_lo, h.hash_lo.p, h.hash_lo.bytes(), 0);
    if (e == cudaSuccess) e = dev_alloc(&c.hash, (nh + 2) * 8);
    if (e == cudaSuccess) e = cudaMemset(c.hash, 0, (nh + 2) * 8);
    if (e == cudaSuccess) { relayout_hash<<<grid, 256>>>((const u32*)r_hi, (const unsigned char*)r_lo, nh, (u64*)c.hash); e = cudaGetLastError(); }
    if (e == cudaSuccess) e = raw(&r_pac, h.pac.p, h.pac.bytes(), 16);
    if (e == cudaSuccess) e = dev_alloc(&c.planes, npw * 8);
    if (e == cudaSuccess) e = cudaMemset(c.planes, 0, npw * 8);
    if (e == cudaSuccess) { relayout_planes<<<grid, 256>>>((const unsigned char*)r_pac, h.N, (n + 31) / 32, (uint2*)c.planes); e = cudaGetLastError(); }
    if (e == cudaSuccess) { c.bytes += h.ssa.bytes(); e = cudaMalloc(&c.ssa, h.ssa.bytes() + 16); }
    if (e == cudaSuccess) e = cudaMemcpy(c.ssa, h.ssa.p, h.ssa.bytes(), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc(&c.chroms, h.chrom_start.size() * 8 + 16);
    if (e == cudaSuccess) e = cudaMemcpy(c.chroms, h.chrom_start.data(), h.chrom_start.size() * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaDeviceSynchronize();
    cudaFree(r_bwt); cudaFree(r_high); cudaFree(r_flag); cudaFree(r_hi); cudaFree(r_lo); cudaFree(r_pac);
    if (e != cudaSuccess) { err_out = std::string("index upload: ") + cudaGetErrorString(e); return; }
    DevIndex& v = c.view;
    v.occ = (const ulonglong2*)c.occ; v.flag = (const ulonglong2*)c.flag; v.hash = (const u64*)c.hash;
    v.ssa = (const u32*)c.ssa; v.planes = (const uint2*)c.planes;
    v.C[0] = h.nacgt[0]; v.C[1] = h.nacgt[1]; v.C[2] = h.nacgt[2];
    v.shapline = h.shapline; v.n_rows = h.sa_length; v.N = h.N;
    v.chrom_start = (const u64*)c.chroms; v.n_chrom = (u32)(h.chrom_start.size() - 1);
    v.dsa_lo = nullptr; v.dsa_hi = nullptr; v.ktab = nullptr; v.kdepth = 0; v.kpow = 1;
    lap("upload + device re-layout");
    // ---- dense suffix array (BMBS_SA=sampled keeps the on-disk 1/8 sampling; default: dense when it fits with room to spare)
    const char* mode = getenv("BMBS_SA");
    // texts of 2^32 rows and more keep bits 32..39 of every suffix-array value in a byte array of their own; BMBS_FORCE_WIDE
    // switches that path on for a small index too (GPU tests: the 5-byte gather and densify's second store run everywhere)
    const bool wide = h.sa_length > 0xFFFFFFFFull || getenv("BMBS_FORCE_WIDE") != nullptr;
    const size_t need = (size_t)h.sa_length * (wide ? 5 : 4);
    size_t free_b = 0, total_b = 0; cudaMemGetInfo(&free_b, &total_b);
    const bool want = mode ? strcmp(mode, "sampled") != 0 : need + (total_b >> 2) < free_b;
    if (want) {
      DeviceCopy& cc = c;
      e = cudaMalloc(&cc.dsa_lo, (size_t)h.sa_length * 4 + 256);
      if (e == cudaSuccess && wide) e = cudaMalloc(&cc.dsa_hi, (size_t)h.sa_length + 256);
      if (e == cudaSuccess) {
        cudaDeviceProp prop; cudaGetDeviceProperties(&prop, cc.dev);
        densify_sa<<<prop.multiProcessorCount * 8, 256>>>(v, (u32*)cc.dsa_lo, (unsigned char*)cc.dsa_hi);
        e = cudaDeviceSynchronize();
      }
      if (e != cudaSuccess) { err_out = std::string("dense suffix array: ") + cudaGetErrorString(e); return; }
      v.dsa_lo = (const u32*)cc.dsa_lo; v.dsa_hi = (const unsigned char*)cc.dsa_hi;
      cudaFree(cc.flag); cudaFree(cc.ssa); cc.flag = nullptr; cc.ssa = nullptr; v.flag = nullptr; v.ssa = nullptr;
      cc.bytes += need; cc.bytes -= nfb * 16 + h.ssa.bytes();
    }
    lap("dense suffix array");
    // ---- deep seed table: K = 16..20 (BMBS_KMER); default: the smallest K whose 3^K exceeds 8 x the text length -- a
    // random K-mer then rarely has a second occurrence, so most seeds end on their first lookup -- if it fits in a quarter of HBM
    {
      int K = 16;
      if (const char* ks = getenv("BMBS_KMER")) K = atoi(ks);
      else { double p = 43046721.0; while (K < 20 && p < 8.0 * (double)n) { p *= 3; ++K; } }
      if (K > 20) K = 20;
      size_t free_b = 0, total_b = 0; cudaMemGetInfo(&free_b, &total_b);
      auto bytes_of = [&](int k) { size_t x = nh ? nh - 1 : 0; for (int i = 16; i < k; ++i) x *= 3; return x * 8; };
      if (!getenv("BMBS_KMER")) while (K > 16 && bytes_of(K) > total_b / 4) --K;
      if (K > 16 && nh > 1) {
        DeviceCopy& cc = c;
        const int D = K - 16; const size_t kb = bytes_of(K);
        e = cudaMalloc(&cc.ktab, kb + 256);
        if (e == cudaSuccess) {
          cudaDeviceProp prop; cudaGetDeviceProperties(&prop, cc.dev);
          const u32 n_keys = (u32)(nh - 1); const int grid = prop.multiProcessorCount * 16;
          if (D == 1) build_ktab<1><<<grid, 128>>>(v, (u64*)cc.ktab, n_keys);
          else if (D == 2) build_ktab<2><<<grid, 128>>>(v, (u64*)cc.ktab, n_keys);
          else if (D == 3) build_ktab<3><<<grid, 128>>>(v, (u64*)cc.ktab, n_keys);
          else build_ktab<4><<<grid, 128>>>(v, (u64*)cc.ktab, n_keys);
          e = cudaDeviceSynchronize();
        }
        if (e != cudaSuccess) { err_out = std::string("deep seed table: ") + cudaGetErrorString(e); return; }
        v.ktab = (const u64*)cc.ktab; v.kdepth = (u32)D; v.kpow = D == 1 ? 3 : D == 2 ? 9 : D == 3 ? 27 : 81;
        cc.bytes += kb;
      }
    }
    lap("deep seed table");
  };
  {
    std::vector<std::thread> th;
    for (int d = 1; d < n_dev; ++d) th.emplace_back(load_on, d);
    load_on(0);
    for (auto& t : th) t.join();
  }
  for (int d = 0; d < n_dev; ++d)
    if (!errors[(size_t)d].empty()) { const std::string m = "device " + std::to_string(devices[d]) + ": " + errors[(size_t)d]; bmbs_index_free(idx); return fail(BMBS_ERR_CUDA, m); }
  *out = idx;
  return BMBS_OK;
}

// ================================================================================================ batch
// what the host reads back after a run and a finish, copied into pinned memory on the batch's stream
struct HostMirror {
  u64 totals[2];                 // BatchView::totals[0..1]: candidate slots, verification work items
  u32 status;                    // BatchView::status
  u64 counters[8];               // BatchView::counters[0..7]
  u64 out_cand;                  // BatchView::totals[3]: out_cand entries of all rounds
  FinCounters fin;
};

struct bmbs_batch {
  bmbs_index* idx = nullptr; const DeviceCopy* copy = nullptr; int dev = 0;
  size_t max_reads = 0, max_bases = 0, cand_cap = 0;
  cudaStream_t stream = nullptr;
  std::vector<void*> allocs;
  BatchView v{};
  char* d_ascii = nullptr; u64* d_offsets = nullptr;
  u64* d_tile = nullptr;
  HostMirror* mirror = nullptr;  // pinned
  cudaEvent_t ev[11] = {nullptr};
  FinishView fv{};               // finishing (bmbs_batch_finish)
  bool finished = false;
  int n_reads = 0, pe = 0, max_len = 0, launches = 0, sm_count = 148, seed_blocks_per_sm = 8; u32 seed_plane_cap = 0;
  u32 seed_grid = 0, verify_grid = 0, verify_block = 0;   // as launched last (bmbs_batch_grid)
  bool ran = false;
};

namespace {
// a finishing kernel over the batch's FinishView (FINISH_PARAMS)
template <class K> void launch_finish(bmbs_batch* b, K kernel, u32 grid, u32 block, size_t smem) {
  const FinishView& f = b->fv;
  kernel<<<grid, block, smem, b->stream>>>(b->copy->view, b->v, f.fin, f.mism, f.mism_cap, f.fb, f.fb_cap, f.sort_list, f.long_list, f.huge_list, f.fc, f.pe_short);
  ++b->launches;
}
// verify_windows over the work list.  Shared memory: five match planes of nch2 overlapping 64-bit chunks per thread; the 32-bit
// band (every k <= 15) reads the chunk of its column only, the 64-bit band the one after it as well.  The grid is what is
// resident at once (the kernel is a grid-stride loop over windows of equal cost: blocks beyond that would run alone at the end).
void launch_verify(bmbs_batch* b, double e_rate, cudaStream_t s, const DevIndex& ix, const BatchView& v) {
  const double kd = e_rate * (double)b->max_len;                       // k of the longest read, as pack_reads computes it
  const int kmax = kd >= 31.0 ? 31 : (int)(u64)kd;
  const int nch2 = (b->max_len + 31) / 32 + (kmax <= 15 ? 0 : 1);
  int bd = 128;
  while (bd > 32 && (size_t)5 * nch2 * bd * 8 > 96 * 1024) bd >>= 1;
  const size_t smem = (size_t)5 * std::max(nch2, 1) * bd * 8;
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, verify_windows, bd, smem) != cudaSuccess || per_sm < 1) per_sm = 1;
  if (per_sm > 12) per_sm = 12;
  verify_windows<<<b->sm_count * per_sm, bd, smem, s>>>(ix, v, std::max(nch2, 1)); ++b->launches;
  b->verify_grid = (u32)(b->sm_count * per_sm); b->verify_block = (u32)bd;
}
// device arrays of a batch are carved out of one slab (one cudaMalloc per batch context): requests are recorded first
struct SlabRequest { void** slot; size_t bytes; };
thread_local std::vector<SlabRequest> g_slab;
template <class T> cudaError_t dalloc(bmbs_batch*, T** p, size_t n) {
  g_slab.push_back({(void**)p, ((n * sizeof(T) + 256) + 255) & ~(size_t)255});
  return cudaSuccess;
}
cudaError_t slab_commit(bmbs_batch* b) {
  size_t total = 0; for (auto& r : g_slab) total += r.bytes;
  void* base = nullptr; cudaError_t e = cudaMalloc(&base, total + 256);
  if (e == cudaSuccess) {
    b->allocs.push_back(base);
    char* p = (char*)base;
    for (auto& r : g_slab) { *r.slot = p; p += r.bytes; }
  }
  g_slab.clear();
  return e;
}
}  // namespace

extern "C" void bmbs_batch_free(bmbs_batch* b) {
  if (!b) return;
  cudaSetDevice(b->dev);
  for (void* p : b->allocs) cudaFree(p);
  if (b->mirror) cudaFreeHost(b->mirror);
  for (auto& e : b->ev) if (e) cudaEventDestroy(e);
  if (b->stream) cudaStreamDestroy(b->stream);
  delete b;
}

extern "C" int bmbs_batch_create(bmbs_index* idx, int dev, size_t max_reads, size_t max_bases, size_t cand_cap, bmbs_batch** out) {
  if (!idx || !out || max_reads == 0) return fail(BMBS_ERR_ARG, "bad argument");
  const DeviceCopy* c = idx->on(dev);
  if (!c) return fail(BMBS_ERR_ARG, "index was not loaded on device " + std::to_string(dev));
  if (cand_cap >= 0xFFFFFFF0ull || max_reads >= 0x7FFFFFF0ull) return fail(BMBS_ERR_ARG, "capacity too large");
  CU(cudaSetDevice(dev));
  bmbs_batch* b = new bmbs_batch();
  b->idx = idx; b->copy = c; b->dev = dev; b->max_reads = max_reads; b->max_bases = max_bases; b->cand_cap = cand_cap;
  b->sm_count = c->grid_sms;
  BatchView& v = b->v;
  const size_t R = max_reads + 2, S = cand_cap + 64;
  g_slab.clear();
  cudaError_t e = cudaStreamCreateWithFlags(&b->stream, cudaStreamNonBlocking);
  auto A = [&](cudaError_t x) { if (e == cudaSuccess) e = x; };
  A(dalloc(b, &b->d_ascii, max_bases + 64)); A(dalloc(b, &b->d_offsets, R));
  A(dalloc(b, &v.codes, 4 * (max_bases / 32 + 2 * R + 64))); A(dalloc(b, &v.rplanes, max_bases / 32 + 2 * R + 64)); A(dalloc(b, &v.len, R)); A(dalloc(b, &v.first_c, R)); A(dalloc(b, &v.kk, R));
  A(dalloc(b, &v.state, R)); A(dalloc(b, &v.flags, R)); A(dalloc(b, &v.one_mm, R)); A(dalloc(b, &v.site0, R));
  A(dalloc(b, &v.list_count, 4));
  A(dalloc(b, &v.bk, 5 * R)); A(dalloc(b, &v.first_cands, R)); A(dalloc(b, &v.list4, R)); A(dalloc(b, &v.res_first, R)); A(dalloc(b, &v.res_n, R));
  A(dalloc(b, &v.ntask, R)); A(dalloc(b, &v.ncand, R)); A(dalloc(b, &v.coff, R)); A(dalloc(b, &v.tasks, (size_t)MAX_TASKS * max_reads));
  A(dalloc(b, &v.slot_row, S)); A(dalloc(b, &v.slot_adj, S)); A(dalloc(b, &v.slot_read, S)); A(dalloc(b, &v.cand, S)); A(dalloc(b, &v.vcnt, S));
  A(dalloc(b, &v.nv, R)); A(dalloc(b, &v.voff, R)); A(dalloc(b, &v.keep, S));
  A(dalloc(b, &v.vitems, S)); A(dalloc(b, &v.out_cand, S));
  A(dalloc(b, &v.out_res, R)); A(dalloc(b, &v.big_list, R)); A(dalloc(b, &v.big_count, 4)); A(dalloc(b, &v.sort32, R)); A(dalloc(b, &v.sort_count, 4)); A(dalloc(b, &v.mid_list, R)); A(dalloc(b, &v.big1k_list, R));
  v.scratch_cap = 2 * S + 65536;
  A(dalloc(b, &v.scratch, (size_t)v.scratch_cap)); A(dalloc(b, &v.scratch_used, 4));
  A(dalloc(b, &v.counters, 16)); A(dalloc(b, &v.totals, 4)); A(dalloc(b, &v.status, 4));
  A(dalloc(b, &b->d_tile, R / SCAN_TILE + 8));
  FinishView& f = b->fv;
  f.mism_cap = (u32)(32 * R);          // a read holds at most 31 mismatch positions
  f.fb_cap = (u32)S;                   // a handed-back read returns its whole slice of out_cand
  A(dalloc(b, &f.fin, R)); A(dalloc(b, &f.mism, f.mism_cap)); A(dalloc(b, &f.fb, f.fb_cap)); A(dalloc(b, &f.sort_list, R)); A(dalloc(b, &f.long_list, R)); A(dalloc(b, &f.huge_list, R)); A(dalloc(b, &f.fc, 1));
  f.pe_short = 48;                     // pairs with more hits go to finish_pe_long (BMBS_PE_FIN_SHORT: tests)
  if (const char* e = getenv("BMBS_PE_FIN_SHORT")) f.pe_short = (u32)std::max(0, atoi(e));
  A(slab_commit(b));
  A(cudaMallocHost((void**)&b->mirror, sizeof(HostMirror)));
  for (auto& evt : b->ev) A(cudaEventCreate(&evt));
  if (e != cudaSuccess) { std::string m = std::string("batch allocation: ") + cudaGetErrorString(e); bmbs_batch_free(b); return fail(BMBS_ERR_CUDA, m); }
  v.slot_cap = cand_cap;
  // verify_windows may need more than 48 KB of dynamic shared memory for long reads
  cudaFuncSetAttribute(verify_windows, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
  cudaFuncSetAttribute(votes_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(BIG_SMEM_ELEMS * sizeof(u64)));
  cudaFuncSetAttribute(finish_pe_long, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(PE_FIN_WARPS * 2 * PE_FIN_STAGE * sizeof(bmbs_cand)));
  *out = b;
  return BMBS_OK;
}

extern "C" int bmbs_batch_upload(bmbs_batch* b, const char* seqs, const uint64_t* offsets, int n_reads, int pe) {
  if (!b || !seqs || !offsets || n_reads < 0) return fail(BMBS_ERR_ARG, "bad argument");
  if ((size_t)n_reads > b->max_reads) return fail(BMBS_ERR_ARG, "batch has more reads than bmbs_batch_create allowed");
  if (pe && (n_reads & 1)) return fail(BMBS_ERR_ARG, "paired batch needs an even number of reads");
  const u64 bases = offsets[n_reads] - offsets[0];
  if (offsets[0] != 0) return fail(BMBS_ERR_ARG, "offsets[0] must be 0");
  if (bases > b->max_bases) return fail(BMBS_ERR_ARG, "batch has more bases than bmbs_batch_create allowed");
  // the longest read (sizes the shared-memory staging of the kernels); a million-read batch passes through here on the caller's
  // thread every step, so: no branch in the loop, four independent maxima, one check at the end (offsets that run backwards
  // wrap to a huge length and fail the same check)
  u64 m0 = 0, m1 = 0, m2 = 0, m3 = 0;
  int i = 0;
  for (; i + 4 <= n_reads; i += 4) {
    const u64 a = offsets[i + 1] - offsets[i], b2 = offsets[i + 2] - offsets[i + 1], c = offsets[i + 3] - offsets[i + 2], d = offsets[i + 4] - offsets[i + 3];
    m0 = a > m0 ? a : m0; m1 = b2 > m1 ? b2 : m1; m2 = c > m2 ? c : m2; m3 = d > m3 ? d : m3;
  }
  for (; i < n_reads; ++i) { const u64 a = offsets[i + 1] - offsets[i]; m0 = a > m0 ? a : m0; }
  const u64 longest = std::max(std::max(m0, m1), std::max(m2, m3));
  if (longest > 1000) return fail(BMBS_ERR_ARG, "read longer than 1000 bases (SEQ_MAX_LENGTH, Auxiliary.h:15)");
  const int max_len = (int)longest;
  CU(cudaSetDevice(b->dev));
  CU(cudaMemcpyAsync(b->d_ascii, seqs, bases, cudaMemcpyHostToDevice, b->stream));
  CU(cudaMemcpyAsync(b->d_offsets, offsets, (size_t)(n_reads + 1) * 8, cudaMemcpyHostToDevice, b->stream));
  b->n_reads = n_reads; b->pe = pe; b->max_len = max_len; b->ran = false; b->finished = false;
  return BMBS_OK;
}

namespace {
int run_scan(bmbs_batch* b, const u32* in, u32 n, u32* out, u64* total, u64 cap, u32 cap_bit, const u64* base = nullptr) {
  const u32 tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
  scan_tiles<<<tiles, SCAN_TILE, 0, b->stream>>>(in, n, b->d_tile, b->v.status);
  scan_tile_sums<<<1, 1024, 0, b->stream>>>(b->d_tile, tiles, total, cap, b->v.status, cap_bit, base);
  scan_apply<<<tiles, SCAN_TILE, 0, b->stream>>>(in, n, b->d_tile, out);
  b->launches += 3;
  return 0;
}

// The candidates of a seeding round, from the seed tasks of every read: offsets of the candidate slots, the sites of the
// seeds' rows, then the votes per read (votes_classify finishes short segments, the other five kernels sort longer ones by
// size class).  `located`, when given, is recorded after expand_locate.
int launch_candidates(bmbs_batch* b, const DevIndex& ix, const BatchView& v, cudaEvent_t located) {
  const int n = v.n_reads;
  cudaStream_t s = b->stream;
  run_scan(b, v.ncand, (u32)n, v.coff, v.totals, v.slot_cap, 2u);
  expand_locate<<<(n + 127) / 128, 128, 0, s>>>(ix, v); ++b->launches;
  if (located) CU(cudaEventRecord(located, s));
  votes_classify<<<(n + 127) / 128, 128, 0, s>>>(v); ++b->launches;
  votes_sort<32><<<b->sm_count * 4, 128, 0, s>>>(v); ++b->launches;
  votes_mid<<<b->sm_count * 8, 128, 0, s>>>(v); ++b->launches;
  votes_big1k<<<b->sm_count * 8, 128, 0, s>>>(v); ++b->launches;
  votes_big<<<b->sm_count * 4, 256, 4096 * sizeof(u64), s>>>(v, 4096u, 0u, 4096u); ++b->launches;
  votes_big<<<b->sm_count * 2, BIG_THREADS, BIG_SMEM_ELEMS * sizeof(u64), s>>>(v, (u32)BIG_SMEM_ELEMS, 8192u, 0xFFFFFFFFu); ++b->launches;
  return BMBS_OK;
}
}  // namespace

extern "C" int bmbs_batch_run(bmbs_batch* b, const bmbs_params* prm) {
  if (!b || !prm) return fail(BMBS_ERR_ARG, "bad argument");
  if (prm->sensitive && !b->pe) return fail(BMBS_ERR_ARG, "sensitive=1 only applies to paired batches (Process_CommandLines.cpp: --sensitive is a --pe mode)");
  CU(cudaSetDevice(b->dev));
  BatchView& v = b->v;
  const int n = b->n_reads;
  v.ascii = b->d_ascii; v.offsets = b->d_offsets; v.n_reads = n; v.pe = b->pe;
  v.e_rate = prm->e_rate; v.seed_len = (u32)prm->seed_len; v.dmax_base = prm->max_ins; v.dmin_base = prm->min_ins;
  v.sensitive = prm->sensitive ? 1 : 0; v.amb_out = prm->ambiguous_out ? 1 : 0; v.round = 0; v.multi_cap = prm->sensitive ? MAX_PE_MULTI_SENSITIVE : MAX_PE_MULTI;
  b->launches = 0;
  cudaStream_t s = b->stream;
  const DevIndex ix = b->copy->view;
  CU(cudaMemsetAsync(v.counters, 0, 16 * 8, s)); CU(cudaMemsetAsync(v.totals, 0, 4 * 8, s)); CU(cudaMemsetAsync(v.status, 0, 16, s));
  CU(cudaMemsetAsync(v.big_count, 0, 16, s)); CU(cudaMemsetAsync(v.scratch_used, 0, 16, s)); CU(cudaMemsetAsync(v.list_count, 0, 16, s));
  CU(cudaMemsetAsync(v.sort_count, 0, 16, s));
  CU(cudaEventRecord(b->ev[0], s));
  if (n > 0) {
    pack_reads<<<(n + 15) / 16, 128, 0, s>>>(v); ++b->launches;
    CU(cudaEventRecord(b->ev[1], s));
    // read chunks staged per thread in shared memory: max_len/32 + 2 chunks of 16 bytes, at most 12 (longer reads: the rest from global memory)
    const u32 plane_cap = (u32)std::min(b->max_len / 32 + 2, 12);
    const size_t seed_smem = (size_t)plane_cap * SEED_BLOCK * sizeof(uint4);
    // one persistent kernel: a lane per read, one dependent access per loop iteration, finished lanes take the next read
    if (plane_cap != b->seed_plane_cap) {      // resident blocks: registers and the staged read chunks decide
      int per_sm = 0;
      if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, seed_reads, SEED_BLOCK, seed_smem) == cudaSuccess && per_sm > 0) b->seed_blocks_per_sm = per_sm;
      if (const char* e = getenv("BMBS_SEED_BLOCKS")) b->seed_blocks_per_sm = std::max(1, atoi(e));
      b->seed_plane_cap = plane_cap;
    }
    const int seed_blocks = std::min((n + SEED_BLOCK - 1) / SEED_BLOCK, b->sm_count * b->seed_blocks_per_sm);
    seed_reads<<<seed_blocks, SEED_BLOCK, seed_smem, s>>>(ix, v, plane_cap); ++b->launches;
    b->seed_grid = (u32)seed_blocks;
    CU(cudaEventRecord(b->ev[2], s));
    if (int rc = launch_candidates(b, ix, v, b->ev[3])) return rc;
    CU(cudaEventRecord(b->ev[4], s));
    if (b->pe && !v.sensitive) { filter_pairs_kernel<<<(n / 2 + 127) / 128, 128, 0, s>>>(v); ++b->launches; }
    CU(cudaEventRecord(b->ev[5], s));
    run_scan(b, v.nv, (u32)n, v.voff, v.totals + 1, v.slot_cap, 4u);
    gather_work<<<(n + 127) / 128, 128, 0, s>>>(v); ++b->launches;
    launch_verify(b, v.e_rate, s, ix, v);
    CU(cudaEventRecord(b->ev[6], s));
    if (v.sensitive) {
      // --pe --sensitive: pair logic on the verified lists, then one re-seeding round for the mates left without a hit
      sens_pair<<<(n / 2 + 3) / 4, 128, 0, s>>>(v); ++b->launches;      // one warp per pair
      reseed_clear<<<(n + 255) / 256, 256, 0, s>>>(v); ++b->launches;
      BatchView w = v; w.round = 1;
      seed_reseed<<<b->sm_count * 8, SEED_BLOCK, seed_smem, s>>>(ix, w, plane_cap); ++b->launches;
      if (int rc = launch_candidates(b, ix, w, nullptr)) return rc;
      sens_reseed_filter<<<b->sm_count * 4, 128, 0, s>>>(w); ++b->launches;
      run_scan(b, w.nv, (u32)n, w.voff, w.totals + 1, w.slot_cap, 4u, w.totals + 2);
      gather_work<<<(n + 127) / 128, 128, 0, s>>>(w); ++b->launches;
      launch_verify(b, w.e_rate, s, ix, w);
      sens_reseed_finish<<<b->sm_count * 4, 128, 0, s>>>(w); ++b->launches;
    }
    CU(cudaEventRecord(b->ev[7], s));
    finalize_reads<<<(n + 255) / 256, 256, 0, s>>>(v); ++b->launches;
  } else {
    for (int i = 1; i <= 7; ++i) CU(cudaEventRecord(b->ev[i], s));
    b->seed_grid = 0;
  }
  CU(cudaEventRecord(b->ev[8], s));
  HostMirror* h = b->mirror;
  CU(cudaMemcpyAsync(h->totals, v.totals, sizeof(h->totals), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&h->out_cand, v.totals + 3, sizeof(h->out_cand), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(&h->status, v.status, sizeof(h->status), cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(h->counters, v.counters, sizeof(h->counters), cudaMemcpyDeviceToHost, s));
  CU(cudaGetLastError());
  b->ran = true; b->finished = false;
  return BMBS_OK;
}

extern "C" int bmbs_batch_finish(bmbs_batch* b) {
  if (!b || !b->ran) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  CU(cudaSetDevice(b->dev));
  cudaStream_t s = b->stream;
  const int n = b->n_reads;
  const FinishView& f = b->fv;
  CU(cudaMemsetAsync(f.fc, 0, sizeof(FinCounters), s));
  CU(cudaEventRecord(b->ev[9], s));
  if (n > 0 && b->pe) {
    launch_finish(b, finish_pe, (n / 2 + 127) / 128, 128, 0);
    const size_t pe_smem = (size_t)PE_FIN_WARPS * 2 * PE_FIN_STAGE * sizeof(bmbs_cand);
    launch_finish(b, finish_pe_long, b->sm_count * 2, 32 * PE_FIN_WARPS, pe_smem);
  } else if (n > 0) {
    launch_finish(b, finish_se, (n + 127) / 128, 128, 0);
    launch_finish(b, finish_huge, b->sm_count * 2, 256, 0);
    launch_finish(b, finish_long, b->sm_count * 12, 128, 0);
    launch_finish(b, finish_sorted, b->sm_count * 6, 32 * FIN_SORT_WARPS, 0);
  }
  CU(cudaEventRecord(b->ev[10], s));
  CU(cudaMemcpyAsync(&b->mirror->fin, f.fc, sizeof(FinCounters), cudaMemcpyDeviceToHost, s));
  CU(cudaGetLastError());
  b->finished = true;
  return BMBS_OK;
}

extern "C" int bmbs_batch_sync(bmbs_batch* b) {
  if (!b) return fail(BMBS_ERR_ARG, "bad argument");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  return BMBS_OK;
}

namespace {
int check_status(bmbs_batch* b, size_t* used) {
  const HostMirror& h = *b->mirror;
  const u32 st = h.status;
  if (used) *used = (size_t)h.out_cand;
  if (st & 1u) return fail(BMBS_ERR_CAPACITY, "a read produced more seed tasks than the per-read table holds");
  if (st & 2u) { if (used) *used = (size_t)h.totals[0]; return fail(BMBS_ERR_CAPACITY, "candidate slots exceed the batch capacity (" + std::to_string(h.totals[0]) + " needed): create the batch with a larger cand_cap or send fewer reads"); }
  if (st & 4u) return fail(BMBS_ERR_CAPACITY, "verification work exceeds the batch capacity");
  if (st & 8u) return fail(BMBS_ERR_CAPACITY, "sort scratch exhausted");
  return BMBS_OK;
}
}  // namespace

extern "C" int bmbs_batch_output_sizes(bmbs_batch* b, size_t* n_cand, size_t* n_mism) {
  if (!b || !b->ran) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  if (n_mism) *n_mism = 0;
  int rc = check_status(b, n_cand);
  if (rc) return rc;
  if (b->finished) { if (n_mism) *n_mism = (size_t)b->mirror->fin.mism_used; if (n_cand) *n_cand = (size_t)b->mirror->fin.fb_used; }
  return BMBS_OK;
}

extern "C" int bmbs_batch_download(bmbs_batch* b, bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap, size_t* cand_used) {
  if (!b || !b->ran || !res) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  int rc = check_status(b, cand_used);
  if (rc) return rc;
  const size_t work = (size_t)b->mirror->out_cand;
  if (work > cand_cap) { if (cand_used) *cand_used = work; return fail(BMBS_ERR_CAPACITY, "caller's cand[] holds " + std::to_string(cand_cap) + " entries, " + std::to_string(work) + " needed"); }
  if (b->n_reads) CU(cudaMemcpyAsync(res, b->v.out_res, (size_t)b->n_reads * sizeof(bmbs_read_result), cudaMemcpyDeviceToHost, b->stream));
  if (work) { if (!cand) return fail(BMBS_ERR_ARG, "cand is null"); CU(cudaMemcpyAsync(cand, b->v.out_cand, work * sizeof(bmbs_cand), cudaMemcpyDeviceToHost, b->stream)); }
  CU(cudaStreamSynchronize(b->stream));
  return BMBS_OK;
}

extern "C" int bmbs_batch_download_final(bmbs_batch* b, bmbs_final* fin, uint16_t* mism, size_t mism_cap, size_t* mism_used,
                                         bmbs_cand* cand, size_t cand_cap, size_t* cand_used) {
  if (!b || !b->ran || !b->finished || !fin) return fail(BMBS_ERR_ARG, "bad argument or batch not finished");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  int rc = check_status(b, cand_used);
  if (rc) return rc;
  const FinishView& f = b->fv;
  const size_t nm = (size_t)b->mirror->fin.mism_used, nfb = (size_t)b->mirror->fin.fb_used;
  if (mism_used) *mism_used = nm;
  if (cand_used) *cand_used = nfb;
  if (nm > f.mism_cap || nfb > f.fb_cap) return fail(BMBS_ERR_CAPACITY, "finishing buffers of the batch are too small");
  if (nm > mism_cap || nfb > cand_cap) return fail(BMBS_ERR_CAPACITY, "caller's mism[] / cand[] too small: " + std::to_string(nm) + " / " + std::to_string(nfb) + " entries needed");
  if (b->n_reads) CU(cudaMemcpyAsync(fin, f.fin, (size_t)b->n_reads * sizeof(bmbs_final), cudaMemcpyDeviceToHost, b->stream));
  if (nm) { if (!mism) return fail(BMBS_ERR_ARG, "mism is null"); CU(cudaMemcpyAsync(mism, f.mism, nm * sizeof(uint16_t), cudaMemcpyDeviceToHost, b->stream)); }
  if (nfb) { if (!cand) return fail(BMBS_ERR_ARG, "cand is null"); CU(cudaMemcpyAsync(cand, f.fb, nfb * sizeof(bmbs_cand), cudaMemcpyDeviceToHost, b->stream)); }
  CU(cudaStreamSynchronize(b->stream));
  return BMBS_OK;
}

extern "C" int bmbs_batch_finish_counters(bmbs_batch* b, uint64_t c[8]) {
  if (!b || !b->finished || !c) return fail(BMBS_ERR_ARG, "bad argument or batch not finished");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  const FinCounters& f = b->mirror->fin;
  c[0] = f.mism_used; c[1] = f.fb_used; c[2] = f.n_sorted; c[3] = f.n_host; c[4] = f.n_dp; c[5] = f.n_unc_idx; c[6] = f.n_unc_sbd;
  float ms = 0; CU(cudaEventElapsedTime(&ms, b->ev[9], b->ev[10]));
  c[7] = (uint64_t)(ms * 1000.0f);
  return BMBS_OK;
}

extern "C" int bmbs_batch_timings(bmbs_batch* b, float ms[8]) {
  if (!b || !b->ran || !ms) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  CU(cudaSetDevice(b->dev));
  CU(cudaEventSynchronize(b->ev[8]));
  CU(cudaEventElapsedTime(&ms[0], b->ev[0], b->ev[8]));
  for (int i = 1; i <= 7; ++i) CU(cudaEventElapsedTime(&ms[i], b->ev[i - 1], b->ev[i]));
  return BMBS_OK;
}

extern "C" int bmbs_batch_counters(bmbs_batch* b, uint64_t c[8]) {
  if (!b || !b->ran || !c) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  CU(cudaSetDevice(b->dev));
  CU(cudaStreamSynchronize(b->stream));
  for (int i = 0; i < 8; ++i) c[i] = b->mirror->counters[i];
  c[CNT_CAND] = b->mirror->totals[0];
  return BMBS_OK;
}

extern "C" int bmbs_batch_launches(bmbs_batch* b) { return b ? b->launches : 0; }

// test entry: the grids as launched, so that a test can see how many items each lane / thread of the persistent and grid-stride
// kernels had to take
extern "C" int bmbs_batch_grid(bmbs_batch* b, uint32_t g[4]) {
  if (!b || !g) return fail(BMBS_ERR_ARG, "bad argument");
  g[0] = (uint32_t)b->sm_count; g[1] = b->seed_grid; g[2] = b->verify_grid; g[3] = b->verify_block;
  return BMBS_OK;
}

extern "C" void* bmbs_pinned_alloc(size_t bytes) { void* p = nullptr; return cudaMallocHost(&p, bytes ? bytes : 1) == cudaSuccess ? p : nullptr; }
extern "C" void bmbs_pinned_free(void* p) { if (p) cudaFreeHost(p); }

// test entry: the order std::sort by vote (descending) leaves lists of <= 2048 votes (each < 32) in, by the warp routine of
// the device finishing (warp_replay_partitions + stable final pass); ok[i] = 0 when the replay gave up (depth limit)
extern "C" int bmbs_debug_sort_order(int dev, const uint32_t* votes, const uint32_t* offsets, uint32_t n_lists, uint16_t* order, int* ok) {
  if (!votes || !offsets || !order || !ok) return fail(BMBS_ERR_ARG, "bad argument");
  CU(cudaSetDevice(dev));
  const size_t total = offsets[n_lists];
  for (uint32_t i = 0; i < n_lists; ++i) if (offsets[i + 1] - offsets[i] > (uint32_t)FIN_SORT_CAP) return fail(BMBS_ERR_ARG, "list longer than the replay capacity");
  u32 *d_v = nullptr, *d_o = nullptr; unsigned short* d_ord = nullptr; int* d_ok = nullptr;
  CU(cudaMalloc(&d_v, total * 4 + 16)); CU(cudaMalloc(&d_o, (size_t)(n_lists + 1) * 4)); CU(cudaMalloc(&d_ord, total * 2 + 16)); CU(cudaMalloc(&d_ok, (size_t)n_lists * 4 + 16));
  CU(cudaMemcpy(d_v, votes, total * 4, cudaMemcpyHostToDevice)); CU(cudaMemcpy(d_o, offsets, (size_t)(n_lists + 1) * 4, cudaMemcpyHostToDevice));
  debug_sort_order<<<148 * 2, 32 * FIN_SORT_WARPS>>>(d_v, d_o, n_lists, d_ord, d_ok);
  CU(cudaDeviceSynchronize());
  CU(cudaMemcpy(order, d_ord, total * 2, cudaMemcpyDeviceToHost)); CU(cudaMemcpy(ok, d_ok, (size_t)n_lists * 4, cudaMemcpyDeviceToHost));
  cudaFree(d_v); cudaFree(d_o); cudaFree(d_ord); cudaFree(d_ok);
  return BMBS_OK;
}

// ================================================================================================ one-call forms
namespace {
struct Cached { bmbs_index* idx; u64 serial; int dev; bmbs_batch* b; };
thread_local std::vector<Cached> g_cache;

int cached_batch(bmbs_index* idx, int dev, size_t reads, size_t bases, size_t cand_cap, bmbs_batch** out) {
  // contexts of indexes that have been freed since: their device slabs are still ours to release (bmbs_batch_free does not
  // touch the index), the entries go
  for (size_t i = 0; i < g_cache.size();) {
    if (g_cache[i].b && serial_live(g_cache[i].serial)) { ++i; continue; }
    if (g_cache[i].b) bmbs_batch_free(g_cache[i].b);
    g_cache[i] = g_cache.back(); g_cache.pop_back();
  }
  for (auto& c : g_cache)
    if (c.idx == idx && c.serial == idx->serial && c.dev == dev) {
      if (c.b->max_reads >= reads && c.b->max_bases >= bases && c.b->cand_cap >= cand_cap) { *out = c.b; return BMBS_OK; }
      bmbs_batch_free(c.b); c.b = nullptr;
      int rc = bmbs_batch_create(idx, dev, reads, bases, cand_cap, &c.b);
      if (rc) { c.idx = nullptr; c.serial = 0; return rc; }
      *out = c.b; return BMBS_OK;
    }
  bmbs_batch* b = nullptr;
  int rc = bmbs_batch_create(idx, dev, reads, bases, cand_cap, &b);
  if (rc) return rc;
  g_cache.push_back({idx, idx->serial, dev, b});
  *out = b; return BMBS_OK;
}

int map_batch(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_reads, int pe, const bmbs_params* prm,
              bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap, size_t* cand_used) {
  if (!idx || !seqs || !offsets || !prm || !res || n_reads < 0) return fail(BMBS_ERR_ARG, "bad argument");
  // device-side slot capacity is the library's business: start from a per-read estimate and grow on overflow;
  // the caller's cand_cap only bounds what is copied back
  size_t dev_cap = (size_t)n_reads * 16 + (1u << 16);
  for (int attempt = 0; attempt < 8; ++attempt) {
    bmbs_batch* b = nullptr;
    int rc = cached_batch(idx, dev, (size_t)n_reads + 1, offsets[n_reads] + 64, dev_cap, &b);
    if (rc) return rc;
    if ((rc = bmbs_batch_upload(b, seqs, offsets, n_reads, pe))) return rc;
    if ((rc = bmbs_batch_run(b, prm))) return rc;
    rc = bmbs_batch_download(b, res, cand, cand_cap, cand_used);
    if (rc == BMBS_ERR_CAPACITY && (b->mirror->status & 2u)) { const size_t slots = (size_t)b->mirror->totals[0]; dev_cap = slots + (slots >> 2) + 1024; continue; }
    return rc;
  }
  return fail(BMBS_ERR_CAPACITY, "candidate slots keep exceeding the device capacity");
}
}  // namespace

extern "C" int bmbs_map_batch_se(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_reads, const bmbs_params* prm,
                                 bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap, size_t* cand_used) {
  return map_batch(idx, dev, seqs, offsets, n_reads, 0, prm, res, cand, cand_cap, cand_used);
}
extern "C" int bmbs_map_batch_pe(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_pairs, const bmbs_params* prm,
                                 bmbs_read_result* res, bmbs_cand* cand, size_t cand_cap, size_t* cand_used) {
  return map_batch(idx, dev, seqs, offsets, 2 * n_pairs, 1, prm, res, cand, cand_cap, cand_used);
}

namespace {
__global__ void verify_setup(BatchView b, const u32* read_idx, const u64* sites, u32 n) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < (u32)b.n_reads) b.state[i] = BMBS_VERIFY;
  if (i < n) {
    const u32 r = read_idx[i];
    VerifyItem it; it.site = sites[i]; it.wi = i; it.vote = 0; it.code_off = code_word_offset(b.offsets, (int)r); it.L = b.len[r]; it.k = b.kk[r]; it.pad = 0;
    b.vitems[i] = it;
  }
  if (i == 0) { b.totals[1] = n; b.totals[3] = n; b.list_count[3] = n; }
}
__global__ void verify_unpack(const bmbs_cand* c, u32 n, int* end_site, u32* err) {
  const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { end_site[i] = c[i].end_site; err[i] = c[i].err == 0xFFFF ? 0xFFFFFFFFu : c[i].err; }
}
}  // namespace

// Kernel 3 alone over the reads of the last bmbs_batch_upload: pack, then one verify_windows launch over n (read, site) items.
extern "C" int bmbs_batch_verify(bmbs_batch* b, const uint32_t* read_idx, const uint64_t* sites, size_t n, double e_rate) {
  if (!b || (n && (!read_idx || !sites))) return fail(BMBS_ERR_ARG, "bad argument");
  if (n > b->cand_cap) return fail(BMBS_ERR_CAPACITY, "more work items than the batch's cand_cap");
  const int n_reads = b->n_reads;
  for (size_t i = 0; i < n; ++i) if (read_idx[i] >= (uint32_t)n_reads) return fail(BMBS_ERR_ARG, "read_idx out of range");
  CU(cudaSetDevice(b->dev));
  BatchView& v = b->v;
  v.ascii = b->d_ascii; v.offsets = b->d_offsets; v.n_reads = n_reads; v.pe = 0; v.e_rate = e_rate; v.sensitive = 0; v.round = 0;
  cudaStream_t s = b->stream;
  CU(cudaMemsetAsync(v.counters, 0, 16 * 8, s)); CU(cudaMemsetAsync(v.totals, 0, 4 * 8, s)); CU(cudaMemsetAsync(v.status, 0, 16, s));
  CU(cudaMemsetAsync(v.list_count, 0, 16, s));
  // stage the work list through slot_read[] / slot_row[] (free in this mode)
  if (n) { CU(cudaMemcpyAsync(v.slot_read, read_idx, n * 4, cudaMemcpyHostToDevice, s)); CU(cudaMemcpyAsync(v.slot_row, sites, n * 8, cudaMemcpyHostToDevice, s)); }
  b->launches = 0;
  CU(cudaEventRecord(b->ev[0], s));
  if (n_reads) { pack_reads<<<(n_reads + 15) / 16, 128, 0, s>>>(v); ++b->launches; }
  const u32 m = (u32)(n > (size_t)n_reads ? n : (size_t)n_reads);
  if (m) { verify_setup<<<(m + 255) / 256, 256, 0, s>>>(v, v.slot_read, v.slot_row, (u32)n); ++b->launches; }
  for (int i = 1; i <= 5; ++i) CU(cudaEventRecord(b->ev[i], s));
  launch_verify(b, v.e_rate, s, b->copy->view, v);
  CU(cudaEventRecord(b->ev[6], s)); CU(cudaEventRecord(b->ev[7], s)); CU(cudaEventRecord(b->ev[8], s));
  HostMirror* h = b->mirror;
  CU(cudaMemcpyAsync(h->counters, v.counters, sizeof(h->counters), cudaMemcpyDeviceToHost, s));
  CU(cudaGetLastError());
  h->totals[0] = 0; h->totals[1] = n; h->out_cand = n; h->status = 0; b->ran = true;
  return BMBS_OK;
}

extern "C" int bmbs_batch_download_verify(bmbs_batch* b, int32_t* end_site, uint32_t* err, size_t n) {
  if (!b || !b->ran || (n && (!end_site || !err))) return fail(BMBS_ERR_ARG, "bad argument or batch not run");
  if (n > b->cand_cap) return fail(BMBS_ERR_ARG, "n exceeds the batch capacity");
  CU(cudaSetDevice(b->dev));
  cudaStream_t s = b->stream;
  // unpack on the device into the (now free) work arrays, then two plain copies
  int* d_end = (int*)b->v.slot_read; u32* d_err = b->v.slot_adj;
  if (n) {
    verify_unpack<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(b->v.out_cand, (u32)n, d_end, d_err);
    CU(cudaMemcpyAsync(end_site, d_end, n * 4, cudaMemcpyDeviceToHost, s));
    CU(cudaMemcpyAsync(err, d_err, n * 4, cudaMemcpyDeviceToHost, s));
  }
  CU(cudaStreamSynchronize(s));
  CU(cudaGetLastError());
  return BMBS_OK;
}

extern "C" int bmbs_verify(bmbs_index* idx, int dev, const char* seqs, const uint64_t* offsets, int n_reads, const uint32_t* read_idx,
                           const uint64_t* sites, size_t n, double e_rate, int32_t* end_site, uint32_t* err) {
  if (!idx || !seqs || !offsets || !read_idx || !sites || !end_site || !err) return fail(BMBS_ERR_ARG, "null argument");
  bmbs_batch* b = nullptr;
  int rc = cached_batch(idx, dev, (size_t)n_reads + 1, offsets[n_reads] + 64, n + 1024, &b);
  if (rc) return rc;
  if ((rc = bmbs_batch_upload(b, seqs, offsets, n_reads, 0))) return rc;
  if ((rc = bmbs_batch_verify(b, read_idx, sites, n, e_rate))) return rc;
  return bmbs_batch_download_verify(b, end_site, err, n);
}

// ================================================================================================ CIGAR refinement
struct bmbs_refiner {
  bmbs_index* idx = nullptr; const DeviceCopy* copy = nullptr; int dev = 0;
  cudaStream_t stream = nullptr;
  // device buffers, grown on demand
  char* d_seq = nullptr; char* d_qual = nullptr; size_t cap_bytes = 0;
  bmbs_refine_item* d_items = nullptr; bmbs_refine_result* d_res = nullptr; u64* d_ops_off = nullptr; size_t cap_items = 0;
  u32* d_ops_scratch = nullptr; u32* d_ops_out = nullptr; size_t cap_ops = 0;
  unsigned long long* d_total = nullptr;
  // page-locked staging for the offsets and the counter
  u64* h_off = nullptr; size_t cap_h_off = 0; unsigned long long* h_total = nullptr;
  int sm_count = 148;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr; bool timed = false;
};

extern "C" int bmbs_refiner_create(bmbs_index* idx, int dev, bmbs_refiner** out) {
  if (!idx || !out) return fail(BMBS_ERR_ARG, "null argument");
  const DeviceCopy* copy = nullptr;
  for (auto& c : idx->copies) if (c.dev == dev) copy = &c;
  if (!copy) return fail(BMBS_ERR_ARG, "the index is not resident on device " + std::to_string(dev));
  CU(cudaSetDevice(dev));
  bmbs_refiner* r = new bmbs_refiner();
  r->idx = idx; r->copy = copy; r->dev = dev;
  CU(cudaStreamCreateWithFlags(&r->stream, cudaStreamNonBlocking));
  r->sm_count = copy->grid_sms;
  cudaFuncSetAttribute(refine_warp<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, RW_WARPS * 1000 * (int)sizeof(uint4));
  cudaFuncSetAttribute(refine_warp<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, RW_WARPS * 1000 * 2 * (int)sizeof(uint4));
  CU(cudaMalloc(&r->d_total, 8));
  CU(cudaMallocHost(&r->h_total, 8));
  CU(cudaEventCreate(&r->ev0)); CU(cudaEventCreate(&r->ev1));
  *out = r;
  return BMBS_OK;
}

extern "C" void bmbs_refiner_free(bmbs_refiner* r) {
  if (!r) return;
  cudaSetDevice(r->dev);
  cudaStreamSynchronize(r->stream);
  cudaFree(r->d_seq); cudaFree(r->d_qual); cudaFree(r->d_items); cudaFree(r->d_res); cudaFree(r->d_ops_off);
  cudaFree(r->d_ops_scratch); cudaFree(r->d_ops_out); cudaFree(r->d_total);
  cudaFreeHost(r->h_off); cudaFreeHost(r->h_total);
  if (r->ev0) cudaEventDestroy(r->ev0); if (r->ev1) cudaEventDestroy(r->ev1);
  cudaStreamDestroy(r->stream);
  delete r;
}

extern "C" int bmbs_refine(bmbs_refiner* r, const char* seqs, const char* quals, size_t bytes, const bmbs_refine_item* items, size_t n,
                           const bmbs_scoring* sc, bmbs_refine_result* res, uint32_t* ops, size_t ops_cap, size_t* ops_used) {
  if (!r || !sc || (n && (!seqs || !quals || !items || !res))) return fail(BMBS_ERR_ARG, "null argument");
  if (ops_used) *ops_used = 0;
  if (n == 0) return BMBS_OK;
  CU(cudaSetDevice(r->dev));
  // per-item scratch: 2L + 2k + 2 ops (the longest possible traceback)
  if (n + 1 > r->cap_h_off) { cudaFreeHost(r->h_off); r->cap_h_off = n + 1 + 1024; CU(cudaMallocHost(&r->h_off, r->cap_h_off * 8)); }
  u64* ops_off = r->h_off;
  u64 ops_total = 0;
  // bands of up to 32 cells go to refine_warp<1>, wider ones (up to 63) to refine_warp<2>
  size_t n_cls[2] = {0, 0}; u32 max_len[2] = {1, 1};
  for (size_t i = 0; i < n; ++i) {
    const bmbs_refine_item& q = items[i];
    if (q.k > 31) return fail(BMBS_ERR_ARG, "k > 31");
    if (q.len == 0 || q.len > 1000) return fail(BMBS_ERR_ARG, "read length outside 1..1000");
    if ((size_t)q.seq_off + q.len > bytes) return fail(BMBS_ERR_ARG, "item reaches past the end of seqs[]");
    const int c = 2 * q.k + 1 > 32;
    ++n_cls[c]; if (q.len > max_len[c]) max_len[c] = q.len;
    ops_off[i] = ops_total;
    ops_total += 2ull * q.len + 2ull * q.k + 2;
  }
  ops_off[n] = ops_total;
  if (ops_total > 0xFFFFFFFFull) return fail(BMBS_ERR_CAPACITY, "too many alignments in one bmbs_refine call");
  if (bytes > r->cap_bytes) { cudaFree(r->d_seq); cudaFree(r->d_qual); r->d_seq = r->d_qual = nullptr; r->cap_bytes = bytes + bytes / 2 + 4096; CU(cudaMalloc(&r->d_seq, r->cap_bytes)); CU(cudaMalloc(&r->d_qual, r->cap_bytes)); }
  if (n + 1 > r->cap_items) {
    cudaFree(r->d_items); cudaFree(r->d_res); cudaFree(r->d_ops_off);
    r->cap_items = n + n / 2 + 1024;
    CU(cudaMalloc(&r->d_items, r->cap_items * sizeof(bmbs_refine_item))); CU(cudaMalloc(&r->d_res, r->cap_items * sizeof(bmbs_refine_result)));
    CU(cudaMalloc(&r->d_ops_off, r->cap_items * 8));
  }
  if (ops_total > r->cap_ops) {
    cudaFree(r->d_ops_scratch); cudaFree(r->d_ops_out); r->d_ops_scratch = r->d_ops_out = nullptr;
    r->cap_ops = (size_t)ops_total + (size_t)ops_total / 2 + 1024;
    CU(cudaMalloc(&r->d_ops_scratch, r->cap_ops * 4)); CU(cudaMalloc(&r->d_ops_out, r->cap_ops * 4));
  }
  cudaStream_t s = r->stream;
  CU(cudaMemcpyAsync(r->d_seq, seqs, bytes, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(r->d_qual, quals, bytes, cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(r->d_items, items, n * sizeof(bmbs_refine_item), cudaMemcpyHostToDevice, s));
  CU(cudaMemcpyAsync(r->d_ops_off, ops_off, (n + 1) * 8, cudaMemcpyHostToDevice, s));
  CU(cudaMemsetAsync(r->d_total, 0, 8, s));
  RefineScoring rs{sc->mp_max, sc->mp_min, sc->n_pen, sc->gap_open, sc->gap_ext, sc->q_base};
  CU(cudaEventRecord(r->ev0, s));
  for (int c = 0; c < 2; ++c) {
    if (!n_cls[c]) continue;
    const size_t smem = (size_t)RW_WARPS * max_len[c] * (c + 1) * sizeof(uint4);
    const unsigned blocks = (unsigned)std::min<size_t>((n_cls[c] + RW_WARPS - 1) / RW_WARPS, (size_t)r->sm_count * 16);
    (c ? refine_warp<2> : refine_warp<1>)<<<blocks, 32 * RW_WARPS, smem, s>>>(r->copy->view, r->d_items, (u32)n, r->d_seq, r->d_qual, rs, r->d_ops_scratch,
                                                                             r->d_ops_off, r->d_res, r->d_ops_out, r->d_total, (u64)r->cap_ops, max_len[c]);
  }
  CU(cudaEventRecord(r->ev1, s)); r->timed = true;
  CU(cudaMemcpyAsync(r->h_total, r->d_total, 8, cudaMemcpyDeviceToHost, s));
  CU(cudaMemcpyAsync(res, r->d_res, n * sizeof(bmbs_refine_result), cudaMemcpyDeviceToHost, s));
  CU(cudaStreamSynchronize(s));
  CU(cudaGetLastError());
  const size_t used = (size_t)*r->h_total;
  if (ops_used) *ops_used = used;
  if (used > ops_cap) return fail(BMBS_ERR_CAPACITY, "ops[] holds " + std::to_string(ops_cap) + " entries, " + std::to_string(used) + " needed");
  if (used) { if (!ops) return fail(BMBS_ERR_ARG, "ops is null"); CU(cudaMemcpyAsync(ops, r->d_ops_out, used * 4, cudaMemcpyDeviceToHost, s)); CU(cudaStreamSynchronize(s)); }
  return BMBS_OK;
}

extern "C" int bmbs_refiner_kernel_ms(bmbs_refiner* r, float* ms) {
  if (!r || !ms || !r->timed) return fail(BMBS_ERR_ARG, "bad argument or nothing refined yet");
  CU(cudaSetDevice(r->dev));
  CU(cudaEventSynchronize(r->ev1));
  CU(cudaEventElapsedTime(ms, r->ev0, r->ev1));
  return BMBS_OK;
}

// ================================================================================================ integer-pipe peak
// Denominator of the verification roofline (SURVEY.md §8d): dependent-free LOP3 + IADD3 streams, 8 independent
// chains per thread, every SM full.  Returns 32-bit integer ALU operations per second.
namespace {
__global__ void __launch_bounds__(256) int_pipe_ubench(u32* out, int iters) {
  u32 a[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) a[i] = threadIdx.x * (i + 1) + blockIdx.x;
  const u32 x = out[0], y = out[1];
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      asm volatile("lop3.b32 %0, %0, %1, %2, 0x96;" : "+r"(a[i]) : "r"(x), "r"(y));
      asm volatile("add.u32 %0, %0, %1;" : "+r"(a[i]) : "r"(y));
    }
  }
  u32 s = 0;
#pragma unroll
  for (int i = 0; i < 8; ++i) s ^= a[i];
  if (s == 0x12345678u) out[2] = s;
}
}  // namespace

extern "C" int bmbs_ubench_int_pipe(int dev, double* ops_per_second) {
  if (!ops_per_second) return fail(BMBS_ERR_ARG, "null argument");
  CU(cudaSetDevice(dev));
  cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, dev));
  u32* d = nullptr; CU(cudaMalloc(&d, 64)); CU(cudaMemset(d, 0, 64));
  cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, iters = 1 << 14;
  int_pipe_ubench<<<blocks, 256>>>(d, 256);
  double best = 0;
  for (int rep = 0; rep < 3; ++rep) {
    CU(cudaEventRecord(e0));
    int_pipe_ubench<<<blocks, 256>>>(d, iters);
    CU(cudaEventRecord(e1)); CU(cudaEventSynchronize(e1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, e0, e1));
    const double ops = (double)blocks * 256 * (double)iters * 16 / (ms / 1000.0);
    if (ops > best) best = ops;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *ops_per_second = best;
  return BMBS_OK;
}

// ================================================================================================ random-sector peak
// What bounds the seeding kernels is not streaming bandwidth but how many independent 32-byte sectors HBM delivers per
// second at random addresses (table entries, occ blocks, suffix-array entries).  This measures that rate: every thread
// keeps 8 independent 256-bit loads in flight at hashed addresses over `bytes` of device memory.
namespace {
// V selects the load instruction (BMBS_UBENCH_VARIANT, experiments on how much DRAM traffic one random sector costs)
template <int V>
__global__ void __launch_bounds__(256) random_sector_ubench(const ulonglong4* __restrict__ buf, u64 n_sectors, int iters, u64* sink) {
  u64 x = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * 0x9E3779B97F4A7C15ull + 0x632BE59BD9B4E019ull;
  u64 acc = 0;
  for (int it = 0; it < iters; ++it) {
    u64 a[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) { x ^= x << 13; x ^= x >> 7; x ^= x << 17; a[i] = x % n_sectors; }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      u64 v0 = 0, v1 = 0, v2 = 0, v3 = 0;
      if (V == 0) asm volatile("ld.global.nc.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 1) asm volatile("ld.global.nc.L2::64B.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 2) asm volatile("ld.global.nc.L2::128B.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 3) asm volatile("ld.global.cv.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 4) asm volatile("ld.global.cg.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 5) asm volatile("ld.global.nc.L1::no_allocate.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 6) asm volatile("ld.global.lu.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      if (V == 7) asm volatile("ld.global.nc.u64 %0, [%1];" : "=l"(v0) : "l"(buf + a[i]));
      if (V == 8) asm volatile("ld.global.nc.L1::no_allocate.L2::evict_first.v4.u64 {%0,%1,%2,%3}, [%4];" : "=l"(v0), "=l"(v1), "=l"(v2), "=l"(v3) : "l"(buf + a[i]));
      acc += v0 ^ v3;
    }
  }
  if (acc == 0x1234567ull) *sink = acc;
}
}  // namespace

extern "C" int bmbs_ubench_random_sectors(int dev, size_t bytes, double* sectors_per_second) {
  if (!sectors_per_second || bytes < (1u << 20)) return fail(BMBS_ERR_ARG, "bad argument");
  CU(cudaSetDevice(dev));
  cudaDeviceProp prop; CU(cudaGetDeviceProperties(&prop, dev));
  void* d = nullptr; CU(cudaMalloc(&d, bytes + 64)); CU(cudaMemset(d, 1, bytes));
  u64* sink = (u64*)d;
  cudaEvent_t e0, e1; CU(cudaEventCreate(&e0)); CU(cudaEventCreate(&e1));
  const int blocks = prop.multiProcessorCount * 8, iters = 64;
  const u64 n_sectors = bytes / 32;
  const int variant = getenv("BMBS_UBENCH_VARIANT") ? atoi(getenv("BMBS_UBENCH_VARIANT")) : 0;
  auto launch = [&](int it) {
    const ulonglong4* q = (const ulonglong4*)d;
    switch (variant) {
      case 1: random_sector_ubench<1><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 2: random_sector_ubench<2><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 3: random_sector_ubench<3><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 4: random_sector_ubench<4><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 5: random_sector_ubench<5><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 6: random_sector_ubench<6><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 7: random_sector_ubench<7><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      case 8: random_sector_ubench<8><<<blocks, 256>>>(q, n_sectors, it, sink); break;
      default: random_sector_ubench<0><<<blocks, 256>>>(q, n_sectors, it, sink); break;
    }
  };
  launch(4);
  double best = 0;
  for (int rep = 0; rep < 3; ++rep) {
    CU(cudaEventRecord(e0));
    launch(iters);
    CU(cudaEventRecord(e1)); CU(cudaEventSynchronize(e1));
    float ms = 0; CU(cudaEventElapsedTime(&ms, e0, e1));
    const double rate = (double)blocks * 256 * iters * 8 / (ms / 1000.0);
    if (rate > best) best = rate;
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *sectors_per_second = best;
  return BMBS_OK;
}
