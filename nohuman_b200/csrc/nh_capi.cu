/*
 * nh_capi.cu — the extern "C" boundary of libnohuman_gpu.so (include/nohuman_gpu.h).
 * Host-side plumbing only: reads hash.k2d / opts.k2d / taxo.k2d unchanged
 * (formats: SURVEY.md Appendix B), keeps the table resident in HBM, owns the
 * per-session device buffers and stream, and sequences the four kernels of
 * nh_kernels.cu.  No CPU classification path exists here.
 */
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>

#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/nohuman_gpu.h"
#include "nh_internal.h"
#include "nh_kernels.cuh"

/* ------------------------------------------------------------------ */
static thread_local char g_err[1024] = "";

int nh_set_error(int code, const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}

#define CUDA_TRY(expr)                                                                     \
  do {                                                                                     \
    cudaError_t _e = (expr);                                                               \
    if (_e != cudaSuccess)                                                                 \
      return nh_set_error(NH_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                          __FILE__, __LINE__);                                             \
  } while (0)

extern "C" int nh_abi_version(void) { return NH_ABI_VERSION; }
extern "C" const char *nh_last_error(void) { return g_err; }

extern "C" int nh_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) {
    cudaGetLastError();
    return 0;
  }
  return n;
}

/* ------------------------------------------------------------------ */
/* database                                                            */

static int read_file(const std::string &path, std::vector<uint8_t> &out, size_t max_bytes) {
  FILE *f = fopen(path.c_str(), "rb");
  if (!f) return nh_set_error(NH_ERR_IO, "cannot open %s", path.c_str());
  struct stat st;
  if (fstat(fileno(f), &st)) {
    fclose(f);
    return nh_set_error(NH_ERR_IO, "cannot stat %s", path.c_str());
  }
  size_t n = (size_t)st.st_size;
  if (n > max_bytes) n = max_bytes;
  out.resize(n);
  if (n && fread(out.data(), 1, n, f) != n) {
    fclose(f);
    return nh_set_error(NH_ERR_IO, "short read on %s", path.c_str());
  }
  fclose(f);
  return NH_OK;
}

static bool file_exists(const std::string &p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode);
}

/* validate_db_directory (src/lib.rs:119-141): the three files in dir or dir/db */
int nh_resolve_db_dir(const char *db_dir, std::string &out) {
  const char *req[3] = {"hash.k2d", "opts.k2d", "taxo.k2d"};
  std::string cands[2] = {std::string(db_dir), std::string(db_dir) + "/db"};
  for (auto &c : cands) {
    bool all = true;
    for (auto r : req) all = all && file_exists(c + "/" + r);
    if (all) {
      out = c;
      return NH_OK;
    }
  }
  return nh_set_error(NH_ERR_IO, "Required files (hash.k2d, opts.k2d, taxo.k2d) not found in %s or %s/db",
                      db_dir, db_dir);
}

/* A handle under construction: every failure path releases it through nh_db_close. */
struct DbCloser {
  void operator()(nh_db *db) const { nh_db_close(db); }
};
using DbPtr = std::unique_ptr<nh_db, DbCloser>;

/* the cell array padded to whole 128-byte lines (zero cells), so a 4-sector group load stays inside the allocation */
static size_t table_bytes(uint64_t capacity) { return ((capacity + 31) / 32) * 128; }

/* A new handle for `device` with everything it keeps on the host, from the opts.k2d and taxo.k2d images and the
 * hash.k2d header {capacity, size, key_bits, value_bits}: info, the taxonomy, and every field of params except the
 * device pointers finish_db sets.  It checks all it reads and makes no CUDA call, so malformed input is reported as
 * such before any device work, on a machine without a GPU too. */
static int parse_db(const void *opts, size_t opts_len, const void *taxo, size_t taxo_len, const uint64_t hdr[4],
                    int device, DbPtr &db) {
  db.reset(new nh_db());
  nh_db_info_t &I = db->info;
  I.device = device;
  /* opts.k2d: raw IndexOptions, up to 64 bytes; older DBs are shorter */
  uint8_t ob[64];
  memset(ob, 0, sizeof ob);
  if (opts_len < 32) return nh_set_error(NH_ERR_IO, "opts.k2d too short (%zu bytes)", opts_len);
  memcpy(ob, opts, opts_len < 64 ? opts_len : 64);
  memcpy(&I.k, ob + 0, 8);
  memcpy(&I.l, ob + 8, 8);
  memcpy(&I.spaced_seed_mask, ob + 16, 8);
  memcpy(&I.toggle_mask, ob + 24, 8);
  I.dna_db = ob[32] ? 1 : 0;
  memcpy(&I.minimum_acceptable_hash_value, ob + 40, 8);
  memcpy(&I.revcom_version, ob + 48, 4);
  /* taxo.k2d */
  const uint8_t *tb = (const uint8_t *)taxo;
  if (taxo_len < 32 || memcmp(tb, "K2TAXDAT", 8))
    return nh_set_error(NH_ERR_IO, "taxo.k2d: bad magic");
  uint64_t node_count, name_len, rank_len;
  memcpy(&node_count, tb + 8, 8);
  memcpy(&name_len, tb + 16, 8);
  memcpy(&rank_len, tb + 24, 8);
  if (node_count == 0 || node_count > (1ULL << 31) ||
      taxo_len < 32 + node_count * 56)
    return nh_set_error(NH_ERR_IO, "taxo.k2d: truncated (%llu nodes)", (unsigned long long)node_count);
  I.node_count = node_count;
  db->h_parent.resize(node_count);
  db->h_ext.resize(node_count);
  db->h_name.assign(node_count, std::string());
  db->h_rank.assign(node_count, std::string());
  const uint64_t names_at = 32 + node_count * 56, ranks_at = names_at + name_len;
  const bool have_strings = name_len < taxo_len && rank_len < taxo_len && ranks_at + rank_len <= taxo_len;
  for (uint64_t i = 0; i < node_count; i++) {
    uint64_t parent, ext;
    memcpy(&parent, tb + 32 + i * 56 + 0, 8);
    memcpy(&ext, tb + 32 + i * 56 + 40, 8);
    if (i > 0 && parent >= i)
      return nh_set_error(NH_ERR_UNSUPPORTED,
                          "taxo.k2d: node %llu has parent %llu (kraken2 taxonomies have parent < child)",
                          (unsigned long long)i, (unsigned long long)parent);
    if (ext > 0xFFFFFFFFULL)
      return nh_set_error(NH_ERR_UNSUPPORTED, "taxo.k2d: external id %llu does not fit 32 bits",
                          (unsigned long long)ext);
    db->h_parent[i] = (uint32_t)parent;
    db->h_ext[i] = (uint32_t)ext;
    if (have_strings && i > 0) {
      uint64_t no, ro;
      memcpy(&no, tb + 32 + i * 56 + 24, 8);
      memcpy(&ro, tb + 32 + i * 56 + 32, 8);
      if (no < name_len) db->h_name[i].assign((const char *)tb + names_at + no, strnlen((const char *)tb + names_at + no, name_len - no));
      if (ro < rank_len) db->h_rank[i].assign((const char *)tb + ranks_at + ro, strnlen((const char *)tb + ranks_at + ro, rank_len - ro));
    }
  }
  db->h_parent[0] = 0;
  /* hash.k2d header */
  I.capacity = hdr[0];
  I.size = hdr[1];
  I.key_bits = hdr[2];
  I.value_bits = hdr[3];
  if (I.key_bits + I.value_bits != 32 || I.value_bits < 1 || I.value_bits > 31)
    return nh_set_error(NH_ERR_IO, "hash.k2d: key_bits %llu + value_bits %llu != 32",
                        (unsigned long long)I.key_bits, (unsigned long long)I.value_bits);
  if (I.capacity == 0 || I.capacity >= (1ULL << 62))
    return nh_set_error(NH_ERR_IO, "hash.k2d: bad capacity");
  if (!I.dna_db) return nh_set_error(NH_ERR_UNSUPPORTED, "protein databases are not supported");
  if (I.l < 1 || I.l > 31 || I.k < I.l)
    return nh_set_error(NH_ERR_UNSUPPORTED, "unsupported k=%llu l=%llu", (unsigned long long)I.k,
                        (unsigned long long)I.l);
  if (I.k - I.l + 1 > NH_MAX_WINDOW)
    return nh_set_error(NH_ERR_UNSUPPORTED, "minimizer window k-l+1=%llu exceeds %d",
                        (unsigned long long)(I.k - I.l + 1), NH_MAX_WINDOW);
  if (I.node_count > (1ULL << I.value_bits))
    return nh_set_error(NH_ERR_IO, "taxonomy has more nodes than value_bits can address");
  NhDbParams &P = db->params;
  P.capacity = I.capacity;
  nh_divisor dv = nh_make_divisor(I.capacity);
  P.mod_m = dv.m;
  P.mod_sh1 = dv.sh1;
  P.mod_sh2 = dv.sh2;
  P.value_bits = (uint32_t)I.value_bits;
  P.value_mask = (uint32_t)((1ULL << I.value_bits) - 1);
  P.k = (int32_t)I.k;
  P.l = (int32_t)I.l;
  P.w = P.k - P.l + 1;
  P.tile_pos = NH_TILE_LMERS - (P.w - 1);
  P.legacy_tile_pos = P.tile_pos;
  P.amb_span = P.l > P.k - 1 ? P.l : P.k - 1;
  P.revcom_version = I.revcom_version;
  const uint64_t lmer_mask = (1ULL << (2 * I.l)) - 1;
  P.seed_mask = I.spaced_seed_mask ? I.spaced_seed_mask : lmer_mask;
  P.toggle = I.toggle_mask & lmer_mask;
  P.min_hash = I.minimum_acceptable_hash_value;
  P.node_count = (uint32_t)I.node_count;
  /* a read can hit at most node_count distinct taxa; k_score_big's shared table holds 16K of them */
  if (I.node_count >= NH_BIG_HASH_SLOTS * 3 / 4) {
    uint32_t slots = 1;
    while (slots < 2 * I.node_count) slots <<= 1;
    P.huge_slots = slots;
  }
  return NH_OK;
}

/* The device side of a handle whose host side is filled in and whose cell array is on its device: the taxonomy
 * arrays, the huge taxon table, the kernels' set-up, and the miss filter once the cells hold the table. */
static int finish_db(nh_db *db, bool cells_ready = true) {
  const size_t taxo_bytes = db->info.node_count * 4;
  NhDbParams &P = db->params;
  CUDA_TRY(cudaSetDevice(db->info.device));
  CUDA_TRY(cudaMalloc(&db->d_parent, taxo_bytes));
  CUDA_TRY(cudaMalloc(&db->d_ext, taxo_bytes));
  CUDA_TRY(cudaMemcpy(db->d_parent, db->h_parent.data(), taxo_bytes, cudaMemcpyHostToDevice));
  CUDA_TRY(cudaMemcpy(db->d_ext, db->h_ext.data(), taxo_bytes, cudaMemcpyHostToDevice));
  if (P.huge_slots) {
    const size_t huge_bytes = ((size_t)2 * P.huge_slots + 4) * 4;
    CUDA_TRY(cudaMalloc(&db->d_huge, huge_bytes));
    CUDA_TRY(cudaMemset(db->d_huge, 0, huge_bytes));
  }
  P.cells = db->d_cells;
  P.parent = db->d_parent;
  P.ext_id = db->d_ext;
  P.huge_table = db->d_huge;
  cudaDeviceProp prop;
  CUDA_TRY(cudaGetDeviceProperties(&prop, db->info.device));
  db->sm_count = prop.multiProcessorCount;
  CUDA_TRY(nh_kernels_init());
  return cells_ready ? nh_db_build_filter(db) : NH_OK;
}

/* The miss filter of the table on db's device (nh_kernels.cu, k_filter_build): capacity / 32 records of 32 bytes,
 * a quarter of the table's size.  Built when the cells are on the device; NH_FILTER=0 turns it off, and a failed
 * allocation only means the kernels run without it. */
int nh_db_build_filter(nh_db *db) {
  const char *e = getenv("NH_FILTER");
  if (e && e[0] == '0') return NH_OK;
  NhDbParams &P = db->params;
  const uint64_t n_blocks = (P.capacity + 31) / 32;
  /* value_bits >= 5: the kernel keeps a chain's cell offset (0..31) in the bits of a compacted key that the value would occupy */
  if (!nh_fused_supported(P) || n_blocks > 0xFFFFFFFFull || P.cells == nullptr || P.value_bits < 5) return NH_OK;
  CUDA_TRY(cudaSetDevice(db->info.device));
  if (!db->d_filter) {
    if (cudaMalloc(&db->d_filter, n_blocks * 32) != cudaSuccess) {
      cudaGetLastError();
      db->d_filter = nullptr;
      return NH_OK;
    }
  }
  nh_launch_filter_build(P, db->d_filter, (uint32_t)n_blocks, nullptr);
  const cudaError_t ce = cudaDeviceSynchronize();
  if (ce != cudaSuccess) return nh_set_error(NH_ERR_CUDA, "building the miss filter failed: %s", cudaGetErrorString(ce));
  db->n_filter_blocks = (uint32_t)n_blocks; /* handed to the kernels in NhScoreParams */
  db->info.filter_bytes = n_blocks * 32;
  return NH_OK;
}

static int select_device(int device) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    cudaGetLastError();
    return nh_set_error(NH_ERR_CUDA, "no CUDA device available (%s); libnohuman_gpu has no CPU path",
                        e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
  }
  if (device < 0 || device >= n) return nh_set_error(NH_ERR_INVALID, "device %d out of range (%d devices)", device, n);
  CUDA_TRY(cudaSetDevice(device));
  return NH_OK;
}

/* db's cell array on the current device: table_bytes(capacity), zeroed */
static int alloc_cells(nh_db *db) {
  const size_t bytes = table_bytes(db->info.capacity);
  const cudaError_t e = cudaMalloc(&db->d_cells, bytes);
  if (e != cudaSuccess) {
    db->d_cells = nullptr;
    cudaGetLastError();
    return nh_set_error(NH_ERR_NOMEM, "cudaMalloc(%zu) for the hash table on device %d failed: %s", bytes,
                        db->info.device, cudaGetErrorString(e));
  }
  db->owns_cells = true;
  CUDA_TRY(cudaMemset(db->d_cells, 0, bytes));
  return NH_OK;
}

/* The cells of hash.k2d (f is positioned after the header) into db->d_cells, streamed through two pinned staging
 * buffers so that the multi-GB table never needs a second host copy: reading one chunk overlaps copying the other. */
static int upload_cells(FILE *f, nh_db *db) {
  const size_t CH = 64u << 20, total = db->info.capacity * 4;
  uint8_t *stage[2] = {nullptr, nullptr};
  cudaEvent_t ev[2] = {nullptr, nullptr};
  cudaStream_t cs = nullptr;
  int rc = NH_OK;
  cudaError_t e = cudaStreamCreate(&cs);
  for (int i = 0; i < 2 && e == cudaSuccess; i++) e = cudaEventCreate(&ev[i]);
  for (int i = 0; i < 2 && e == cudaSuccess && rc == NH_OK; i++)
    if (cudaHostAlloc(&stage[i], CH, cudaHostAllocDefault) != cudaSuccess) {
      stage[i] = nullptr;
      cudaGetLastError();
      rc = nh_set_error(NH_ERR_NOMEM, "pinned staging allocation failed");
    }
  size_t done = 0;
  for (int slot = 0; e == cudaSuccess && rc == NH_OK && done < total; slot ^= 1) {
    const size_t n = total - done < CH ? total - done : CH;
    if ((e = cudaEventSynchronize(ev[slot])) != cudaSuccess) break; /* the copy out of this buffer has finished */
    if (fread(stage[slot], 1, n, f) != n) {
      rc = nh_set_error(NH_ERR_IO, "hash.k2d: short read");
      break;
    }
    if ((e = cudaMemcpyAsync((uint8_t *)db->d_cells + done, stage[slot], n, cudaMemcpyHostToDevice, cs)) != cudaSuccess ||
        (e = cudaEventRecord(ev[slot], cs)) != cudaSuccess)
      break;
    done += n;
  }
  if (cs) {
    const cudaError_t se = cudaStreamSynchronize(cs); /* no copy may still read a staging buffer when it is freed */
    if (e == cudaSuccess) e = se;
  }
  for (int i = 0; i < 2; i++) {
    if (stage[i]) cudaFreeHost(stage[i]);
    if (ev[i]) cudaEventDestroy(ev[i]);
  }
  if (cs) cudaStreamDestroy(cs);
  if (rc == NH_OK && e != cudaSuccess) rc = nh_set_error(NH_ERR_CUDA, "table upload failed: %s", cudaGetErrorString(e));
  return rc;
}

extern "C" int nh_db_open_memory(const void *opts, size_t opts_len, const void *taxo, size_t taxo_len,
                                 const uint64_t hash_header[4], const uint32_t *cells,
                                 int cells_on_device, int device, nh_db **out) {
  if (!opts || !taxo || !hash_header || !cells || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  DbPtr db;
  int rc = parse_db(opts, opts_len, taxo, taxo_len, hash_header, device, db);
  if (!rc) rc = select_device(device);
  if (rc) return rc;
  if (cells_on_device) {
    if (((uintptr_t)cells & 127u) != 0) return nh_set_error(NH_ERR_INVALID, "device cell array must be 128-byte aligned");
    db->d_cells = const_cast<uint32_t *>(cells); /* adopted: the caller keeps ownership */
  } else {
    if ((rc = alloc_cells(db.get()))) return rc;
    const cudaError_t e = cudaMemcpy(db->d_cells, cells, db->info.capacity * 4, cudaMemcpyHostToDevice);
    if (e != cudaSuccess)
      return nh_set_error(NH_ERR_CUDA, "copying the hash table to the device failed: %s", cudaGetErrorString(e));
  }
  if ((rc = finish_db(db.get()))) return rc;
  *out = db.release();
  return NH_OK;
}

/* value_bits as build_db.cc picks it: the smallest b with 2^b >= node_count, read here from taxo.k2d's header,
 * which parse_db then checks with the rest of the image */
int nh_db_create_empty(const void *opts, size_t opts_len, const void *taxo, size_t taxo_len,
                       uint64_t capacity, int device, nh_db **out) {
  uint64_t node_count = 0, vb = 1;
  if (taxo_len >= 16) memcpy(&node_count, (const uint8_t *)taxo + 8, 8);
  while (vb < 31 && (1ULL << vb) < node_count) vb++;
  const uint64_t hdr[4] = {capacity, 0, 32 - vb, vb};
  DbPtr db;
  int rc = parse_db(opts, opts_len, taxo, taxo_len, hdr, device, db);
  if (!rc) rc = select_device(device);
  if (!rc) rc = alloc_cells(db.get());
  if (!rc) rc = finish_db(db.get(), false);
  if (rc) return rc;
  *out = db.release();
  return NH_OK;
}

extern "C" int nh_db_open(const char *db_dir, int device, nh_db **out) {
  if (!db_dir || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  std::string dir;
  std::vector<uint8_t> opts, taxo;
  int rc = nh_resolve_db_dir(db_dir, dir);
  if (!rc) rc = read_file(dir + "/opts.k2d", opts, 64);
  if (!rc) rc = read_file(dir + "/taxo.k2d", taxo, (size_t)-1);
  if (rc) return rc;
  /* hash.k2d: 32-byte header, then capacity x u32 */
  const std::string hp = dir + "/hash.k2d";
  std::unique_ptr<FILE, int (*)(FILE *)> f(fopen(hp.c_str(), "rb"), fclose);
  if (!f) return nh_set_error(NH_ERR_IO, "cannot open %s", hp.c_str());
  uint64_t hdr[4];
  if (fread(hdr, 8, 4, f.get()) != 4) return nh_set_error(NH_ERR_IO, "hash.k2d: short header");
  struct stat st;
  if (fstat(fileno(f.get()), &st)) return nh_set_error(NH_ERR_IO, "cannot stat %s", hp.c_str());
  if ((uint64_t)st.st_size != 32 + hdr[0] * 4)
    return nh_set_error(NH_ERR_IO, "hash.k2d: size %lld != 32 + 4*capacity(%llu)", (long long)st.st_size,
                        (unsigned long long)hdr[0]);
  DbPtr db;
  rc = parse_db(opts.data(), opts.size(), taxo.data(), taxo.size(), hdr, device, db);
  if (!rc) rc = select_device(device);
  if (!rc) rc = alloc_cells(db.get());
  if (!rc) rc = upload_cells(f.get(), db.get());
  if (!rc) rc = finish_db(db.get());
  if (rc) return rc;
  *out = db.release();
  return NH_OK;
}

/* a replica of src on `device`: the same host side, and a zeroed table for the caller to fill and then finish_db */
static int db_replica(const nh_db *src, int device, DbPtr &db) {
  int rc = select_device(device);
  if (rc) return rc;
  db.reset(new nh_db());
  db->info = src->info;
  db->info.device = device;
  db->params = src->params; /* finish_db points it at the replica's own device arrays */
  db->h_parent = src->h_parent;
  db->h_ext = src->h_ext;
  db->h_name = src->h_name;
  db->h_rank = src->h_rank;
  return alloc_cells(db.get());
}

extern "C" int nh_db_clone(const nh_db *src, int device, nh_db **out) {
  if (!src || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  DbPtr db;
  int rc = db_replica(src, device, db);
  if (rc) return rc;
  int can = 0;
  if (cudaDeviceCanAccessPeer(&can, device, src->info.device) == cudaSuccess && can) {
    cudaError_t pe = cudaDeviceEnablePeerAccess(src->info.device, 0);
    if (pe != cudaSuccess) cudaGetLastError(); /* already enabled is fine; the copy works either way */
  }
  const cudaError_t e = cudaMemcpyPeer(db->d_cells, device, src->d_cells, src->info.device, table_bytes(src->info.capacity));
  if (e != cudaSuccess)
    return nh_set_error(NH_ERR_CUDA, "replicating the hash table to device %d failed: %s", device, cudaGetErrorString(e));
  if ((rc = finish_db(db.get()))) return rc;
  *out = db.release();
  return NH_OK;
}

/* ------------------------------------------------------------------ */
/* one disk read, N replicas: NCCL broadcast over NVLink / NVSwitch        */

/* NCCL is bound at run time (libnccl.so.2 is in the image; a process that already loaded torch's
 * copy gets that one): no link-time dependency, and a box without it still gets the peer-copy tree */
namespace {
typedef struct ncclComm *nccl_comm_t;
struct Nccl {
  void *h = nullptr;
  int (*CommInitAll)(nccl_comm_t *, int, const int *) = nullptr;
  int (*CommDestroy)(nccl_comm_t) = nullptr;
  int (*GroupStart)(void) = nullptr;
  int (*GroupEnd)(void) = nullptr;
  int (*Broadcast)(const void *, void *, size_t, int /* ncclDataType_t */, int, nccl_comm_t, cudaStream_t) = nullptr;
  const char *(*GetErrorString)(int) = nullptr;
  bool load() {
    const char *off = getenv("NH_DB_REPLICATE");
    if (off && !strcmp(off, "p2p")) return false;
    h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_LOCAL);
    if (!h) return false;
    CommInitAll = (decltype(CommInitAll))dlsym(h, "ncclCommInitAll");
    CommDestroy = (decltype(CommDestroy))dlsym(h, "ncclCommDestroy");
    GroupStart = (decltype(GroupStart))dlsym(h, "ncclGroupStart");
    GroupEnd = (decltype(GroupEnd))dlsym(h, "ncclGroupEnd");
    Broadcast = (decltype(Broadcast))dlsym(h, "ncclBroadcast");
    GetErrorString = (decltype(GetErrorString))dlsym(h, "ncclGetErrorString");
    return CommInitAll && CommDestroy && GroupStart && GroupEnd && Broadcast && GetErrorString;
  }
};
}  // namespace

extern "C" int nh_db_open_multi(const char *db_dir, const int *device_ids, int n_devices, nh_db **out) {
  if (!db_dir || !device_ids || !out || n_devices < 1) return nh_set_error(NH_ERR_INVALID, "bad argument");
  for (int i = 0; i < n_devices; i++)
    for (int j = 0; j < i; j++)
      if (device_ids[i] == device_ids[j]) return nh_set_error(NH_ERR_INVALID, "device %d listed twice", device_ids[i]);
  for (int i = 0; i < n_devices; i++) out[i] = nullptr;
  int rc = nh_db_open(db_dir, device_ids[0], &out[0]); /* the only disk read */
  if (rc || n_devices == 1) return rc;
  std::vector<DbPtr> dbs((size_t)n_devices);
  dbs[0].reset(out[0]);
  out[0] = nullptr;
  for (int i = 1; i < n_devices; i++)
    if ((rc = db_replica(dbs[0].get(), device_ids[i], dbs[(size_t)i])) != NH_OK) return rc;
  const size_t bytes = table_bytes(dbs[0]->info.capacity);
  std::vector<cudaStream_t> streams((size_t)n_devices, nullptr);
  cudaError_t e = cudaSuccess;
  for (int i = 0; i < n_devices && e == cudaSuccess; i++)
    if ((e = cudaSetDevice(device_ids[i])) == cudaSuccess)
      e = cudaStreamCreateWithFlags(&streams[(size_t)i], cudaStreamNonBlocking);
  int how = 0;
  Nccl nccl;
  if (e == cudaSuccess && nccl.load()) {
    std::vector<nccl_comm_t> comms((size_t)n_devices, nullptr);
    int nr = nccl.CommInitAll(comms.data(), n_devices, device_ids);
    if (nr == 0) {
      nccl.GroupStart();
      for (int i = 0; i < n_devices && nr == 0; i++) {
        cudaSetDevice(device_ids[i]);
        nr = nccl.Broadcast(dbs[0]->d_cells, dbs[(size_t)i]->d_cells, bytes, 1 /* ncclUint8 */, 0, comms[(size_t)i], streams[(size_t)i]);
      }
      const int ge = nccl.GroupEnd();
      if (nr == 0) nr = ge;
      for (int i = 0; i < n_devices; i++) {
        cudaSetDevice(device_ids[i]);
        if (cudaStreamSynchronize(streams[(size_t)i]) != cudaSuccess && nr == 0) nr = -1;
      }
      for (auto c : comms)
        if (c) nccl.CommDestroy(c);
    }
    if (nr == 0) how = 1;
    else cudaGetLastError(); /* fall through to the peer copies */
  }
  if (e == cudaSuccess && !how) {
    /* binomial tree of peer copies: round r doubles the number of replicas (3 rounds for 8 GPUs),
     * every copy of a round on its own stream so they run side by side over NVSwitch */
    for (int have = 1; have < n_devices && e == cudaSuccess; have *= 2) {
      for (int i = 0; i < have && have + i < n_devices; i++) {
        const int src = i, dst = have + i;
        int can = 0;
        cudaSetDevice(device_ids[dst]);
        if (cudaDeviceCanAccessPeer(&can, device_ids[dst], device_ids[src]) == cudaSuccess && can)
          if (cudaDeviceEnablePeerAccess(device_ids[src], 0) != cudaSuccess) cudaGetLastError();
        e = cudaMemcpyPeerAsync(dbs[(size_t)dst]->d_cells, device_ids[dst], dbs[(size_t)src]->d_cells, device_ids[src], bytes,
                                streams[(size_t)dst]);
        if (e != cudaSuccess) break;
      }
      for (int i = 0; i < have && have + i < n_devices; i++) {
        cudaSetDevice(device_ids[have + i]);
        const cudaError_t se = cudaStreamSynchronize(streams[(size_t)(have + i)]);
        if (e == cudaSuccess) e = se;
      }
    }
    how = 2;
  }
  for (int i = 0; i < n_devices; i++)
    if (streams[(size_t)i]) {
      cudaSetDevice(device_ids[i]);
      cudaStreamDestroy(streams[(size_t)i]);
    }
  if (e != cudaSuccess) return nh_set_error(NH_ERR_CUDA, "replicating the hash table failed: %s", cudaGetErrorString(e));
  for (int i = 1; i < n_devices; i++) {
    if ((rc = finish_db(dbs[(size_t)i].get())) != NH_OK) return rc;
    dbs[(size_t)i]->info.replicated_by = how;
  }
  for (int i = 0; i < n_devices; i++) out[i] = dbs[(size_t)i].release();
  return NH_OK;
}

extern "C" int nh_db_info(const nh_db *db, nh_db_info_t *out) {
  if (!db || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  *out = db->info;
  return NH_OK;
}

extern "C" const uint32_t *nh_db_device_cells(const nh_db *db) { return db ? db->d_cells : nullptr; }

extern "C" void nh_db_close(nh_db *db) {
  if (!db) return;
  /* a handle that failed before its device work owns no device memory, and closing it makes no CUDA call */
  void *owned[] = {db->owns_cells ? db->d_cells : nullptr, db->d_parent, db->d_ext, db->d_huge, db->d_filter};
  for (void *p : owned)
    if (p) {
      cudaSetDevice(db->info.device);
      cudaFree(p);
    }
  delete db;
}

/* ------------------------------------------------------------------ */
/* session                                                             */

template <typename T>
static cudaError_t dmalloc(T **p, size_t n) {
  return cudaMalloc((void **)p, n * sizeof(T));
}

/* need_lookups: also allocate the per-lookup scratch of the warp-per-tile kernels (8 + 2 + 4 bytes
 * per base).  The streaming kernel keeps its lookups in shared memory, so ordinary sessions only
 * carry 2 + 4 bytes per base when the caller asked for per-read hit runs (emit_runs). */
int nh_session_create_ex(nh_db *db, const nh_params_t *params, bool need_lookups, nh_session **out) {
  if (!db || !params || !out) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (!(params->confidence >= 0.0 && params->confidence <= 1.0))
    return nh_set_error(NH_ERR_INVALID, "Confidence score must be between 0 and 1");
  CUDA_TRY(cudaSetDevice(db->info.device));
  nh_session *s = new nh_session();
  s->db = db;
  s->params = *params;
  if (s->params.minimum_hit_groups < 0) s->params.minimum_hit_groups = 2;
  if (s->params.threads <= 0) s->params.threads = 1;
  uint64_t mb = params->max_batch_bases ? params->max_batch_bases : (256ULL << 20);
  if (mb > (1ULL << 31)) {
    delete s;
    return nh_set_error(NH_ERR_INVALID, "max_batch_bases must be <= 2^31");
  }
  uint64_t ms = params->max_batch_seqs ? params->max_batch_seqs : mb / 64 + 1024;
  if (ms > (1ULL << 31)) ms = 1ULL << 31;
  if (params->paired) ms += ms & 1;
  s->cap_bases = mb;
  s->cap_seqs = ms;
  {
    /* NH_LEGACY_KERNELS=1 forces the warp-per-tile kernels (A/B runs; databases whose window is not 5 take them anyway) */
    const char *legacy = getenv("NH_LEGACY_KERNELS");
    s->use_fused = nh_fused_supported(db->params) && !(legacy && legacy[0] == '1');
    /* NH_TEST_LANE_TAXA=n shrinks the in-warp taxon table so tests reach the overflow pass */
    const char *lt = getenv("NH_TEST_LANE_TAXA");
    int v = lt ? atoi(lt) : NH_LANE_TAXA;
    s->lane_taxa = v < 1 ? 1 : (v > NH_LANE_TAXA ? NH_LANE_TAXA : v);
    /* NH_FILTER_MODE — who asks the miss filter before the table: 0 nobody, 1 units none of whose lookups has hit so
     * far, 2 every lookup, 3 (default) units whose last few lookups all missed */
    const char *fm = getenv("NH_FILTER_MODE");
    s->filter_mode = fm ? atoi(fm) : 3;
    if (s->filter_mode < 0 || s->filter_mode > 3) s->filter_mode = 3;
    /* NH_FUSED_TILE_POS=n fixes the tile size of the streaming kernel (default: by mean read length) */
    const char *tp = getenv("NH_FUSED_TILE_POS");
    s->forced_tile_pos = tp ? atoi(tp) : 0;
    if (s->forced_tile_pos && s->forced_tile_pos < 16) s->forced_tile_pos = 16;
    if (s->forced_tile_pos > NH_FUSED_TILE_POS_MAX) s->forced_tile_pos = NH_FUSED_TILE_POS_MAX;
  }
  s->P = db->params; /* the session's own copy: enqueue_batch sets the tile size per batch */
  const NhDbParams &P = s->P;
  /* every sequence has at most ceil(positions / tile_pos) tiles; sized for the smallest tile any
   * kernel of this session may use */
  int min_tile = db->params.tile_pos < NH_FUSED_TILE_POS_LONG ? db->params.tile_pos : NH_FUSED_TILE_POS_LONG;
  /* packed input rounds a forced tile size down to a multiple of 32 (enqueue_batch): size for that */
  if (s->forced_tile_pos) min_tile = std::min(min_tile, std::max(32, s->forced_tile_pos & ~31));
  if (s->forced_tile_pos && s->forced_tile_pos < min_tile) min_tile = s->forced_tile_pos;
  if (!s->use_fused || need_lookups) min_tile = std::min(min_tile, (int)db->params.tile_pos);
  s->cap_tiles = ms + mb / (uint64_t)min_tile + 1;
  s->cap_lookups = mb; /* one lookup per k-mer position at most */
  const bool want_lookups = need_lookups || !s->use_fused;
  cudaError_t e = cudaSuccess;
#define ALLOC(ptr, n)                                     \
  if (e == cudaSuccess) e = dmalloc(&(ptr), (size_t)(n)); \
  if (e == cudaSuccess) s->device_bytes += (size_t)(n) * sizeof(*(ptr));
  ALLOC(s->d_bases, mb + 64);
  ALLOC(s->d_offsets, ms + 1);
  ALLOC(s->d_tile_base, ms + 2);
  ALLOC(s->d_seq_info, ms + 1);
  ALLOC(s->d_block_sums, ms / 1024 + 2);
  ALLOC(s->d_tiles, s->cap_tiles);
  ALLOC(s->d_tile_out, s->cap_tiles);
  if (want_lookups) {
    ALLOC(s->d_lk_min, s->cap_lookups);
  }
  if (want_lookups || params->emit_runs) {
    ALLOC(s->d_lk_cnt, s->cap_lookups);
    ALLOC(s->d_lk_taxon, s->cap_lookups);
  }
  ALLOC(s->d_out_call, ms);
  ALLOC(s->d_out_keep, ms);
  ALLOC(s->d_dbg_call, ms);
  ALLOC(s->d_dbg_total, ms);
  ALLOC(s->d_dbg_groups, ms);
  ALLOC(s->d_overflow, ms);
  ALLOC(s->d_deferred, ms);
  ALLOC(s->d_counters, 1);
  if (s->use_fused) {
    ALLOC(s->d_tile_tab, s->cap_tiles);
    ALLOC(s->d_tile_sum, s->cap_tiles);
  }
  if (params->emit_runs) {
    ALLOC(s->d_run_ext, s->cap_lookups);
    ALLOC(s->d_run_len, s->cap_lookups);
    ALLOC(s->d_tile_run_off, s->cap_tiles);
    ALLOC(s->d_run_cursor, 1);
  }
#undef ALLOC
  if (e == cudaSuccess) e = cudaHostAlloc(&s->h_counters, sizeof(NhCounters), cudaHostAllocDefault);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking);
  for (int i = 0; i < NH_NUM_EVENTS && e == cudaSuccess; i++) e = cudaEventCreate(&s->ev[i]);
  if (e == cudaSuccess) e = cudaMemset(s->d_counters, 0, sizeof(NhCounters));
  if (e != cudaSuccess) {
    int rc = nh_set_error(e == cudaErrorMemoryAllocation ? NH_ERR_NOMEM : NH_ERR_CUDA,
                          "session allocation failed: %s", cudaGetErrorString(e));
    nh_session_destroy(s);
    return rc;
  }
  memset(s->h_counters, 0, sizeof(NhCounters));
  (void)P;
  *out = s;
  return NH_OK;
}

extern "C" int nh_session_create(nh_db *db, const nh_params_t *params, nh_session **out) {
  return nh_session_create_ex(db, params, false, out);
}

extern "C" void nh_session_destroy(nh_session *s) {
  if (!s) return;
  cudaSetDevice(s->db->info.device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  cudaFree(s->d_bases);
  cudaFree(s->d_offsets);
  cudaFree(s->d_tile_base);
  cudaFree(s->d_seq_info);
  cudaFree(s->d_block_sums);
  cudaFree(s->d_tiles);
  cudaFree(s->d_tile_out);
  cudaFree(s->d_lk_min);
  cudaFree(s->d_lk_cnt);
  cudaFree(s->d_lk_taxon);
  cudaFree(s->d_out_call);
  cudaFree(s->d_out_keep);
  cudaFree(s->d_dbg_call);
  cudaFree(s->d_dbg_total);
  cudaFree(s->d_dbg_groups);
  cudaFree(s->d_overflow);
  cudaFree(s->d_deferred);
  cudaFree(s->d_counters);
  cudaFree(s->d_tile_tab);
  cudaFree(s->d_tile_sum);
  cudaFree(s->d_run_ext);
  cudaFree(s->d_run_len);
  cudaFree(s->d_tile_run_off);
  cudaFree(s->d_run_cursor);
  cudaFree(s->d_codes);
  cudaFree(s->d_valid);
  cudaFree(s->d_poff);
  nh_pack_pool_destroy(s->pack_pool); /* joins the packer threads */
  if (s->h_codes) cudaFreeHost(s->h_codes);
  if (s->h_valid) cudaFreeHost(s->h_valid);
  if (s->h_poff) cudaFreeHost(s->h_poff);
  if (s->h_len32) cudaFreeHost(s->h_len32);
  cudaFree(s->d_len32);
  cudaFree(s->d_len_sums);
  if (s->ev_block) cudaEventDestroy(s->ev_block);
  if (s->h_counters) cudaFreeHost(s->h_counters);
  for (int i = 0; i < NH_NUM_EVENTS; i++)
    if (s->ev[i]) cudaEventDestroy(s->ev[i]);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;
}

extern "C" void *nh_session_stream(nh_session *s) { return s ? (void *)s->stream : nullptr; }

extern "C" void *nh_host_alloc(size_t bytes) {
  void *p = nullptr;
  if (cudaHostAlloc(&p, bytes, cudaHostAllocPortable) != cudaSuccess) { /* usable from every device */
    cudaGetLastError();
    nh_set_error(NH_ERR_NOMEM, "cudaHostAlloc(%zu) failed", bytes);
    return nullptr;
  }
  return p;
}

extern "C" void nh_host_free(void *p) {
  if (p) cudaFreeHost(p);
}

/* Enqueue the four stages for a batch whose inputs are already on the device. */
static int enqueue_batch(nh_session *s, const uint8_t *d_bases, const uint64_t *d_offsets,
                         uint64_t n_seqs, uint64_t total_bases, uint32_t *d_out_call,
                         uint8_t *d_out_keep, bool with_debug, const uint64_t *d_pos_off,
                         uint64_t *d_pos_min, uint8_t *d_pos_amb) {
  /* Tile size of the streaming kernel: 508 positions keep every short read (2x300 bp included) in
   * one tile; batches of long reads take 252, which doubles the number of 32-tile groups the
   * persistent warps draw from (better balance) at 7 % more overlap scanned. */
  if (s->use_fused) {
    const uint64_t mean_len = n_seqs ? total_bases / n_seqs : 0;
    s->P.tile_pos = s->forced_tile_pos ? s->forced_tile_pos : (mean_len > 1000 ? NH_FUSED_TILE_POS_LONG : NH_FUSED_TILE_POS);
    if (s->packed_next) s->P.tile_pos = std::max(32, s->P.tile_pos & ~31); /* tiles of packed input start on a unit of 32 bases */
  }
  const NhDbParams &P = s->P;
  NhBatchPtrs B;
  memset(&B, 0, sizeof B);
  B.bases = d_bases;
  B.offsets = d_offsets;
  if (s->packed_next) {
    B.codes = s->d_codes;
    B.valid = s->d_valid;
    B.poff = s->d_poff;
  }
  B.n_seqs = (uint32_t)n_seqs;
  B.paired = s->params.paired ? 1 : 0;
  B.n_units = (uint32_t)(B.paired ? n_seqs / 2 : n_seqs);
  B.tile_base = s->d_tile_base;
  B.block_sums = s->d_block_sums;
  B.tiles = s->d_tiles;
  B.tile_out = s->d_tile_out;
  B.lk_min = s->d_lk_min;
  B.lk_cnt = s->d_lk_cnt;
  B.lk_taxon = s->d_lk_taxon;
  B.out_call = d_out_call;
  B.out_keep = d_out_keep;
  if (with_debug) {
    B.dbg_call = s->d_dbg_call;
    B.dbg_total_kmers = s->d_dbg_total;
    B.dbg_hit_groups = s->d_dbg_groups;
  }
  B.overflow_units = s->d_overflow;
  B.counters = s->d_counters;
  B.dbg_pos_offsets = d_pos_off;
  B.dbg_pos_min = d_pos_min;
  B.dbg_pos_ambig = d_pos_amb;
  NhScoreParams SP;
  SP.confidence = s->params.confidence;
  SP.min_hit_groups = s->params.minimum_hit_groups;
  SP.keep_human = s->params.keep_human;
  SP.lane_taxa = s->lane_taxa;
  SP.filter_mode = s->filter_mode;
  SP.filter = s->db->n_filter_blocks ? s->db->d_filter : nullptr;
  SP.n_filter_blocks = s->db->n_filter_blocks;
  const int sm = s->db->sm_count;
  uint64_t tiles_upper = n_seqs + total_bases / (uint64_t)P.tile_pos + 1;
  if (tiles_upper > s->cap_tiles) /* cannot happen for batches within the session's capacity; never write past the tile arrays */
    return nh_set_error(NH_ERR_CAPACITY, "batch needs %llu tiles of %d positions, session holds %llu",
                        (unsigned long long)tiles_upper, (int)P.tile_pos, (unsigned long long)s->cap_tiles);
  uint64_t lookups_upper = total_bases;
  int launches = 0;
  cudaStream_t st = s->stream;
  cudaEventRecord(s->ev[EV_PLAN0], st);
  const bool fused = s->use_fused;
  B.deferred_units = fused ? s->d_deferred : nullptr;
  const bool emit = s->params.emit_runs && d_pos_min == nullptr;
  B.emit_all_taxa = emit ? 1 : 0;
  /* batches of long reads (more than 4 tiles per sequence on average): descriptors written per tile */
  B.tiles_upper = (uint32_t)tiles_upper;
  B.seq_info = tiles_upper > 4 * n_seqs ? s->d_seq_info : nullptr;
  launches += nh_launch_plan(P, B, st);
  cudaEventRecord(s->ev[EV_MIN0], st);
  if (fused) {
    /* scan + probe + in-warp scoring in one kernel; ms_probe reads 0 */
    s->last_form = 2;
    B.tile_tab = s->d_tile_tab;
    B.tile_sum = s->d_tile_sum;
    launches += nh_launch_stream(P, B, SP, (uint32_t)tiles_upper, sm, st);
    cudaEventRecord(s->ev[EV_PROBE0], st);
  } else {
    launches += nh_launch_minimizers(P, B, (uint32_t)tiles_upper, sm, st);
    cudaEventRecord(s->ev[EV_PROBE0], st);
    launches += nh_launch_probe(P, s->d_lk_min, s->d_lk_taxon, &s->d_counters->n_lookups,
                                (uint32_t)lookups_upper, sm, st);
  }
  cudaEventRecord(s->ev[EV_SCORE0], st);
  launches += nh_launch_score(P, B, SP, sm, st);
  if (emit)
    launches += nh_launch_gather_runs(P, B, (uint32_t)tiles_upper, s->d_run_ext, s->d_run_len, s->d_tile_run_off,
                                      s->d_run_cursor, sm, st);
  cudaEventRecord(s->ev[EV_SCORE1], st);
  cudaMemcpyAsync(s->h_counters, s->d_counters, sizeof(NhCounters), cudaMemcpyDeviceToHost, st);
  s->last_launches = (uint32_t)launches;
  s->last_fused = fused;
  s->last_units = B.n_units;
  s->last_seqs = n_seqs;
  s->last_bases = total_bases;
  s->pending = true;
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return nh_set_error(NH_ERR_CUDA, "kernel launch failed: %s", cudaGetErrorString(e));
  return NH_OK;
}

static int check_batch_args(nh_session *s, uint64_t n_seqs, uint64_t total_bases) {
  if (s->params.paired && (n_seqs & 1))
    return nh_set_error(NH_ERR_INVALID, "paired session needs an even number of sequences");
  if (n_seqs > s->cap_seqs)
    return nh_set_error(NH_ERR_CAPACITY, "batch has %llu sequences, session capacity is %llu",
                        (unsigned long long)n_seqs, (unsigned long long)s->cap_seqs);
  if (total_bases > s->cap_bases)
    return nh_set_error(NH_ERR_CAPACITY, "batch has %llu bases, session capacity is %llu",
                        (unsigned long long)total_bases, (unsigned long long)s->cap_bases);
  return NH_OK;
}

extern "C" int nh_session_sync(nh_session *s, nh_batch_stats_t *stats) {
  if (!s) return nh_set_error(NH_ERR_INVALID, "null session");
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (s->pending && s->h_counters->error)
    return nh_set_error(NH_ERR_CUDA, "internal error: a unit's taxon table overflowed although it can hold the whole taxonomy");
  if (stats) {
    memset(stats, 0, sizeof *stats);
    if (s->pending) {
      const NhCounters &c = *s->h_counters;
      stats->n_units = s->last_units;
      stats->n_classified = c.n_classified;
      stats->n_unclassified = s->last_units - c.n_classified;
      stats->n_kept = c.n_kept;
      stats->n_bases = s->last_bases;
      stats->n_tiles = c.n_tiles;
      stats->n_lookups = c.n_lookups;
      stats->n_sector_reads = c.n_sector_reads;
      cudaEventElapsedTime(&stats->ms_plan, s->ev[EV_PLAN0], s->ev[EV_MIN0]);
      cudaEventElapsedTime(&stats->ms_minimizer, s->ev[EV_MIN0], s->ev[EV_PROBE0]);
      cudaEventElapsedTime(&stats->ms_probe, s->ev[EV_PROBE0], s->ev[EV_SCORE0]);
      cudaEventElapsedTime(&stats->ms_score, s->ev[EV_SCORE0], s->ev[EV_SCORE1]);
      if (s->timed_copies) {
        cudaEventElapsedTime(&stats->ms_h2d, s->ev[EV_H2D0], s->ev[EV_PLAN0]);
        cudaEventElapsedTime(&stats->ms_d2h, s->ev[EV_SCORE1], s->ev[EV_D2H1]);
      }
      stats->gpu_launches = s->last_launches;
      stats->fused_kernel = s->last_fused ? (uint32_t)s->last_form : 0u;
    }
  }
  return NH_OK;
}

extern "C" int nh_classify_batch_device(nh_session *s, const uint8_t *d_bases,
                                        const uint64_t *d_offsets, uint64_t n_seqs,
                                        uint64_t total_bases, uint32_t *d_out_call,
                                        uint8_t *d_out_keep) {
  if (!s || !d_bases || !d_offsets) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (((uintptr_t)d_bases & 15u) != 0) /* the streaming kernel stages bases with 16-byte asynchronous copies */
    return nh_set_error(NH_ERR_INVALID, "d_bases must be 16-byte aligned");
  int rc = check_batch_args(s, n_seqs, total_bases);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  s->timed_copies = false;
  if (n_seqs == 0) {
    s->pending = false;
    return NH_OK;
  }
  return enqueue_batch(s, d_bases, d_offsets, n_seqs, total_bases, d_out_call, d_out_keep, false,
                       nullptr, nullptr, nullptr);
}

extern "C" int nh_classify_batch(nh_session *s, const uint8_t *bases, const uint64_t *offsets,
                                 uint64_t n_seqs, uint32_t *out_call, uint8_t *out_keep,
                                 nh_batch_stats_t *stats) {
  if (!s || !offsets || (!bases && n_seqs && offsets[n_seqs] > 0))
    return nh_set_error(NH_ERR_INVALID, "null argument");
  const uint64_t total = n_seqs ? offsets[n_seqs] - offsets[0] : 0;
  if (n_seqs && offsets[0] != 0) return nh_set_error(NH_ERR_INVALID, "offsets[0] must be 0");
  int rc = check_batch_args(s, n_seqs, total);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  if (n_seqs == 0) {
    s->pending = false;
    if (stats) memset(stats, 0, sizeof *stats);
    return NH_OK;
  }
  cudaStream_t st = s->stream;
  const uint64_t n_units = s->params.paired ? n_seqs / 2 : n_seqs;
  cudaEventRecord(s->ev[EV_H2D0], st);
  if (total) CUDA_TRY(cudaMemcpyAsync(s->d_bases, bases, total, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(s->d_offsets, offsets, (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
  rc = enqueue_batch(s, s->d_bases, s->d_offsets, n_seqs, total, s->d_out_call, s->d_out_keep, true,
                     nullptr, nullptr, nullptr);
  if (rc) return rc;
  if (out_call) CUDA_TRY(cudaMemcpyAsync(out_call, s->d_out_call, n_units * 4, cudaMemcpyDeviceToHost, st));
  if (out_keep) CUDA_TRY(cudaMemcpyAsync(out_keep, s->d_out_keep, n_units, cudaMemcpyDeviceToHost, st));
  cudaEventRecord(s->ev[EV_D2H1], st);
  s->timed_copies = true;
  return nh_session_sync(s, stats);
}

static int ensure_packed_planes(nh_session *s, uint64_t cap_units) {
  if (s->d_codes) return NH_OK; /* allocated on the first packed batch */
  cudaError_t e = cudaMalloc(&s->d_codes, cap_units * 8 + 64);
  if (e == cudaSuccess) e = cudaMalloc(&s->d_valid, cap_units * 4 + 64);
  if (e == cudaSuccess) e = cudaMalloc(&s->d_poff, (s->cap_seqs + 1) * 4);
  if (e != cudaSuccess) return nh_set_error(NH_ERR_NOMEM, "allocating the packed input planes failed: %s", cudaGetErrorString(e));
  s->device_bytes += cap_units * 12 + 128 + (s->cap_seqs + 1) * 4;
  return NH_OK;
}

/* Packed host input: 2-bit codes + validity bits + unit offsets (nh_pack_reads) instead of ASCII.
 * 0.4 bytes per base cross PCIe; the kernel instantiation that reads the planes also skips the
 * ASCII -> 2-bit step. */
/* len32 != nullptr: the per-sequence metadata travels as 4-byte lengths and the device rebuilds offsets and
 * first units (nh_classify_batch_pack); otherwise poff and offsets are copied as they are */
static int classify_packed_impl(nh_session *s, const uint8_t *codes, const uint32_t *valid, const uint32_t *poff,
                                const uint64_t *offsets, const uint32_t *len32, uint64_t n_seqs, uint32_t *out_call,
                                uint8_t *out_keep, nh_batch_stats_t *stats) {
  if (!s || !offsets || !poff || (n_seqs && offsets[n_seqs] > 0 && (!codes || !valid)))
    return nh_set_error(NH_ERR_INVALID, "null argument");
  if (!s->use_fused) return nh_set_error(NH_ERR_UNSUPPORTED, "packed input needs the streaming kernel (window of 5 l-mers)");
  if (s->params.emit_runs) return nh_set_error(NH_ERR_UNSUPPORTED, "packed input is not available to sessions created with emit_runs");
  const uint64_t total = n_seqs ? offsets[n_seqs] - offsets[0] : 0;
  if (n_seqs && offsets[0] != 0) return nh_set_error(NH_ERR_INVALID, "offsets[0] must be 0");
  int rc = check_batch_args(s, n_seqs, total);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  if (n_seqs == 0) {
    s->pending = false;
    if (stats) memset(stats, 0, sizeof *stats);
    return NH_OK;
  }
  const uint64_t units = poff[n_seqs];
  const uint64_t cap_units = s->cap_bases / 32 + s->cap_seqs + 1;
  if (units > cap_units) return nh_set_error(NH_ERR_CAPACITY, "packed batch has %llu units, session holds %llu", (unsigned long long)units, (unsigned long long)cap_units);
  rc = ensure_packed_planes(s, cap_units);
  if (rc) return rc;
  cudaStream_t st = s->stream;
  const uint64_t n_units = s->params.paired ? n_seqs / 2 : n_seqs;
  cudaEventRecord(s->ev[EV_H2D0], st);
  if (units) {
    CUDA_TRY(cudaMemcpyAsync(s->d_codes, codes, units * 8, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->d_valid, valid, units * 4, cudaMemcpyHostToDevice, st));
  }
  uint32_t extra_launches = 0;
  if (len32) {
    if (!s->d_len32) {
      cudaError_t e = cudaMalloc(&s->d_len32, (s->cap_seqs + 1) * 4);
      if (e == cudaSuccess) e = cudaMalloc(&s->d_len_sums, (s->cap_seqs / 1024 + 2) * 16);
      if (e != cudaSuccess) return nh_set_error(NH_ERR_NOMEM, "allocating the length scan failed: %s", cudaGetErrorString(e));
      s->device_bytes += (s->cap_seqs + 1) * 4 + (s->cap_seqs / 1024 + 2) * 16;
    }
    CUDA_TRY(cudaMemcpyAsync(s->d_len32, len32, n_seqs * 4, cudaMemcpyHostToDevice, st));
    extra_launches = (uint32_t)nh_launch_len_scan(s->d_len32, (uint32_t)n_seqs, s->d_len_sums, s->d_offsets, s->d_poff, st);
  } else {
    CUDA_TRY(cudaMemcpyAsync(s->d_poff, poff, (n_seqs + 1) * 4, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(s->d_offsets, offsets, (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
  }
  s->packed_next = true;
  rc = enqueue_batch(s, nullptr, s->d_offsets, n_seqs, total, s->d_out_call, s->d_out_keep, true, nullptr, nullptr, nullptr);
  s->packed_next = false;
  if (rc) return rc;
  s->last_launches += extra_launches;
  if (out_call) CUDA_TRY(cudaMemcpyAsync(out_call, s->d_out_call, n_units * 4, cudaMemcpyDeviceToHost, st));
  if (out_keep) CUDA_TRY(cudaMemcpyAsync(out_keep, s->d_out_keep, n_units, cudaMemcpyDeviceToHost, st));
  cudaEventRecord(s->ev[EV_D2H1], st);
  s->timed_copies = true;
  /* sleep until the results are back instead of spinning: callers of the packed entry points run several
   * sessions on host threads whose cores are busy packing the next batches */
  if (!s->ev_block) CUDA_TRY(cudaEventCreateWithFlags(&s->ev_block, cudaEventDisableTiming | cudaEventBlockingSync));
  CUDA_TRY(cudaEventRecord(s->ev_block, st));
  CUDA_TRY(cudaEventSynchronize(s->ev_block));
  return nh_session_sync(s, stats);
}

extern "C" int nh_classify_batch_packed(nh_session *s, const uint8_t *codes, const uint32_t *valid, const uint32_t *poff,
                                        const uint64_t *offsets, uint64_t n_seqs, uint32_t *out_call, uint8_t *out_keep,
                                        nh_batch_stats_t *stats) {
  return classify_packed_impl(s, codes, valid, poff, offsets, nullptr, n_seqs, out_call, out_keep, stats);
}

/* ------------------------------------------------------------------ */
/* per-stage entry points for the parity tests                          */

/* ---- nh_classify_batch_pack: ASCII host input, sent in the packed format ----
 * nh_pack_reads + nh_classify_batch_packed in one call: a pool of `pack_threads` packer threads that lives with
 * the session fills the session's own pinned planes (non-temporal stores: the next reader is the copy engine),
 * three large copies follow, and the calling thread sleeps until the results are back.  Several sessions on as
 * many host threads keep the cores packing while other sessions' copies and kernels run (bench.py `e2e`).
 * A finer-grained pipeline — chunks packed into a ring of cache-resident staging slots and copied one by one —
 * was built and measured slower (56-66 against 76-84 Gbp/s): with every core streaming reads, copies out of the
 * slots ran at 34 GB/s instead of 52 (DESIGN.md §4c). */
struct NhPackPool {
  std::vector<std::thread> threads;
  std::mutex mu;
  std::condition_variable cv_job, cv_done;
  uint64_t generation = 0;
  int running = 0;
  bool quit = false;
  std::function<void(int)> job;

  explicit NhPackPool(int n) {
    for (int t = 0; t < n; t++)
      threads.emplace_back([this, t] {
        uint64_t seen = 0;
        for (;;) {
          std::function<void(int)> fn;
          {
            std::unique_lock<std::mutex> lk(mu);
            cv_job.wait(lk, [&] { return quit || generation != seen; });
            if (quit) return;
            seen = generation;
            fn = job;
          }
          fn(t);
          {
            std::lock_guard<std::mutex> lk(mu);
            if (--running == 0) cv_done.notify_all();
          }
        }
      });
  }
  void run(std::function<void(int)> fn) { /* on every thread of the pool; returns when all are done */
    std::unique_lock<std::mutex> lk(mu);
    job = std::move(fn);
    running = (int)threads.size();
    generation++;
    cv_job.notify_all();
    cv_done.wait(lk, [&] { return running == 0; });
  }
  ~NhPackPool() {
    {
      std::lock_guard<std::mutex> lk(mu);
      quit = true;
    }
    cv_job.notify_all();
    for (auto &t : threads) t.join();
  }
};

void nh_pack_pool_destroy(NhPackPool *p) { delete p; }

extern "C" int nh_classify_batch_pack(nh_session *s, const uint8_t *bases, const uint64_t *offsets, uint64_t n_seqs,
                                      int pack_threads, uint32_t *out_call, uint8_t *out_keep, nh_batch_stats_t *stats) {
  if (!s || !offsets || (!bases && n_seqs && offsets[n_seqs] > 0)) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (!s->use_fused) return nh_set_error(NH_ERR_UNSUPPORTED, "packed input needs the streaming kernel (window of 5 l-mers)");
  if (s->params.emit_runs) return nh_set_error(NH_ERR_UNSUPPORTED, "packed input is not available to sessions created with emit_runs");
  const uint64_t total = n_seqs ? offsets[n_seqs] - offsets[0] : 0;
  if (n_seqs && offsets[0] != 0) return nh_set_error(NH_ERR_INVALID, "offsets[0] must be 0");
  int rc = check_batch_args(s, n_seqs, total);
  if (rc) return rc;
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  if (n_seqs == 0) {
    s->pending = false;
    if (stats) memset(stats, 0, sizeof *stats);
    return NH_OK;
  }
  const uint64_t cap_units = s->cap_bases / 32 + s->cap_seqs + 1;
  const int T = pack_threads < 1 ? 1 : pack_threads > 256 ? 256 : pack_threads;
  if (!s->pack_pool || s->pack_threads != T) {
    nh_pack_pool_destroy(s->pack_pool);
    s->pack_pool = new NhPackPool(T);
    s->pack_threads = T;
  }
  if (!s->h_codes) { /* pinned planes for a whole batch, allocated on the first call */
    cudaError_t e = cudaMallocHost(&s->h_codes, cap_units * 8 + 64);
    if (e == cudaSuccess) e = cudaMallocHost(&s->h_valid, cap_units * 4 + 64);
    if (e == cudaSuccess) e = cudaMallocHost(&s->h_poff, (s->cap_seqs + 1) * 4);
    if (e == cudaSuccess) e = cudaMallocHost(&s->h_len32, (s->cap_seqs + 1) * 4);
    if (e != cudaSuccess) return nh_set_error(NH_ERR_NOMEM, "pinned planes for the packed batch: %s", cudaGetErrorString(e));
  }
  /* units per thread range; prefix over the ranges; unit offsets and the planes of every range */
  std::vector<uint64_t> part((size_t)T + 1, 0);
  auto range = [&](int t, uint64_t *a, uint64_t *b) {
    *a = n_seqs * (uint64_t)t / (uint64_t)T;
    *b = n_seqs * (uint64_t)(t + 1) / (uint64_t)T;
  };
  s->pack_pool->run([&](int t) {
    uint64_t a, b, u = 0;
    range(t, &a, &b);
    for (uint64_t q = a; q < b; q++) u += (offsets[q + 1] - offsets[q] + 31) >> 5;
    part[(size_t)t + 1] = u;
  });
  for (int t = 0; t < T; t++) part[(size_t)t + 1] += part[(size_t)t];
  const uint64_t units = part[(size_t)T];
  if (units > cap_units || units > 0xFFFFFFFFull)
    return nh_set_error(NH_ERR_CAPACITY, "packed batch has %llu units, session holds %llu", (unsigned long long)units, (unsigned long long)cap_units);
  uint32_t *h_poff = s->h_poff, *h_len32 = s->h_len32;
  std::atomic<int> too_long{0};
  s->pack_pool->run([&](int t) {
    uint64_t a, b;
    range(t, &a, &b);
    uint64_t u = part[(size_t)t];
    for (uint64_t q = a; q < b; q++) {
      const uint64_t len = offsets[q + 1] - offsets[q];
      if (len > 0xFFFFFFFFull) too_long.store(1);
      h_poff[q] = (uint32_t)u;
      h_len32[q] = (uint32_t)len;
      u += (len + 31) >> 5;
    }
    nh_pack_range(bases, offsets, total, a, b, s->h_codes, s->h_valid, h_poff);
  });
  h_poff[n_seqs] = (uint32_t)units;
  /* 4 bytes per sequence cross PCIe (lengths); the device rebuilds offsets and first units */
  static const bool send_offsets = getenv("NH_PACK_SEND_OFFSETS") != nullptr; /* A/B switch: 12 bytes per sequence as before */
  return classify_packed_impl(s, s->h_codes, s->h_valid, h_poff, offsets, too_long.load() || send_offsets ? nullptr : h_len32, n_seqs,
                              out_call, out_keep, stats);
}

extern "C" int nh_debug_minimizers(nh_session *s, const uint8_t *bases, const uint64_t *offsets,
                                   uint64_t n_seqs, const uint64_t *pos_offsets, uint64_t *out_min,
                                   uint8_t *out_ambig) {
  if (!s || !offsets || !pos_offsets || !out_min || !out_ambig)
    return nh_set_error(NH_ERR_INVALID, "null argument");
  if (n_seqs == 0) return NH_OK;
  const uint64_t total = offsets[n_seqs];
  int rc = check_batch_args(s, n_seqs & ~(uint64_t)(s->params.paired ? 1 : 0), total);
  if (rc) return rc;
  if (s->params.paired && (n_seqs & 1)) return nh_set_error(NH_ERR_INVALID, "odd sequence count");
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  const uint64_t npos = pos_offsets[n_seqs];
  uint64_t *d_pos_off = nullptr, *d_min = nullptr;
  uint8_t *d_amb = nullptr;
  CUDA_TRY(cudaMalloc(&d_pos_off, (n_seqs + 1) * 8));
  CUDA_TRY(cudaMalloc(&d_min, (npos + 1) * 8));
  CUDA_TRY(cudaMalloc(&d_amb, npos + 1));
  cudaStream_t st = s->stream;
  if (total) CUDA_TRY(cudaMemcpyAsync(s->d_bases, bases, total, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(s->d_offsets, offsets, (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemcpyAsync(d_pos_off, pos_offsets, (n_seqs + 1) * 8, cudaMemcpyHostToDevice, st));
  CUDA_TRY(cudaMemsetAsync(d_min, 0xEE, (npos + 1) * 8, st));
  CUDA_TRY(cudaMemsetAsync(d_amb, 0xEE, npos + 1, st));
  rc = enqueue_batch(s, s->d_bases, s->d_offsets, n_seqs, total, s->d_out_call, s->d_out_keep, true,
                     d_pos_off, d_min, d_amb);
  if (rc == NH_OK) {
    cudaMemcpyAsync(out_min, d_min, npos * 8, cudaMemcpyDeviceToHost, st);
    cudaMemcpyAsync(out_ambig, d_amb, npos, cudaMemcpyDeviceToHost, st);
    s->timed_copies = false;
    rc = nh_session_sync(s, nullptr);
  }
  cudaFree(d_pos_off);
  cudaFree(d_min);
  cudaFree(d_amb);
  return rc;
}

extern "C" int nh_debug_probe(nh_session *s, const uint64_t *keys, uint64_t n, uint32_t *out_taxon) {
  if (!s || !keys || !out_taxon) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (n == 0) return NH_OK;
  if (n > 0xFFFFFFFFULL) return nh_set_error(NH_ERR_CAPACITY, "too many keys");
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  uint64_t *d_keys = nullptr;
  uint32_t *d_tax = nullptr;
  CUDA_TRY(cudaMalloc(&d_keys, n * 8));
  CUDA_TRY(cudaMalloc(&d_tax, n * 4));
  cudaStream_t st = s->stream;
  CUDA_TRY(cudaMemcpyAsync(d_keys, keys, n * 8, cudaMemcpyHostToDevice, st));
  nh_launch_probe(s->db->params, d_keys, d_tax, nullptr, (uint32_t)n, s->db->sm_count, st);
  CUDA_TRY(cudaMemcpyAsync(out_taxon, d_tax, n * 4, cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  cudaFree(d_keys);
  cudaFree(d_tax);
  return NH_OK;
}

extern "C" int nh_debug_last_batch(nh_session *s, uint32_t *out_call_internal,
                                   uint32_t *out_total_kmers, uint32_t *out_hit_groups,
                                   uint64_t n_units) {
  if (!s) return nh_set_error(NH_ERR_INVALID, "null session");
  if (n_units > s->last_units) return nh_set_error(NH_ERR_INVALID, "last batch had fewer units");
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  if (out_call_internal)
    CUDA_TRY(cudaMemcpy(out_call_internal, s->d_dbg_call, n_units * 4, cudaMemcpyDeviceToHost));
  if (out_total_kmers)
    CUDA_TRY(cudaMemcpy(out_total_kmers, s->d_dbg_total, n_units * 4, cudaMemcpyDeviceToHost));
  if (out_hit_groups)
    CUDA_TRY(cudaMemcpy(out_hit_groups, s->d_dbg_groups, n_units * 4, cudaMemcpyDeviceToHost));
  return NH_OK;
}

extern "C" int nh_last_batch_runs(nh_session *s, uint64_t n_seqs, uint32_t *seq_first_run,
                                  uint32_t *run_taxon_ext, uint16_t *run_len, uint64_t run_capacity,
                                  uint64_t *n_runs) {
  if (!s || !seq_first_run || !run_taxon_ext || !run_len) return nh_set_error(NH_ERR_INVALID, "null argument");
  if (!s->params.emit_runs) return nh_set_error(NH_ERR_INVALID, "session was not created with emit_runs");
  if (n_seqs != s->last_seqs) return nh_set_error(NH_ERR_INVALID, "last batch had %llu sequences", (unsigned long long)s->last_seqs);
  CUDA_TRY(cudaSetDevice(s->db->info.device));
  CUDA_TRY(cudaStreamSynchronize(s->stream));
  const uint32_t n_tiles = s->h_counters->n_tiles;
  uint32_t total = 0;
  CUDA_TRY(cudaMemcpy(&total, s->d_run_cursor, 4, cudaMemcpyDeviceToHost));
  if (n_runs) *n_runs = total;
  if (total > run_capacity) return nh_set_error(NH_ERR_CAPACITY, "%u runs do not fit the caller's %llu", total, (unsigned long long)run_capacity);
  std::vector<uint32_t> tile_base(n_seqs + 1), tile_off(n_tiles), ext(total);
  std::vector<NhTileOut> tile_out(n_tiles);
  std::vector<uint16_t> len(total);
  CUDA_TRY(cudaMemcpy(tile_base.data(), s->d_tile_base, (n_seqs + 1) * 4, cudaMemcpyDeviceToHost));
  if (n_tiles) {
    CUDA_TRY(cudaMemcpy(tile_off.data(), s->d_tile_run_off, (size_t)n_tiles * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(tile_out.data(), s->d_tile_out, (size_t)n_tiles * sizeof(NhTileOut), cudaMemcpyDeviceToHost));
  }
  if (total) {
    CUDA_TRY(cudaMemcpy(ext.data(), s->d_run_ext, (size_t)total * 4, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(len.data(), s->d_run_len, (size_t)total * 2, cudaMemcpyDeviceToHost));
  }
  /* tiles were packed in completion order; hand the runs back in sequence order */
  uint32_t o = 0;
  for (uint64_t i = 0; i < n_seqs; i++) {
    seq_first_run[i] = o;
    for (uint32_t t = tile_base[i]; t < tile_base[i + 1]; t++) {
      const uint32_t n = tile_out[t].lk_cnt, from = tile_off[t];
      memcpy(run_taxon_ext + o, ext.data() + from, (size_t)n * 4);
      memcpy(run_len + o, len.data() + from, (size_t)n * 2);
      o += n;
    }
  }
  seq_first_run[n_seqs] = o;
  return NH_OK;
}

/* ------------------------------------------------------------------ */
extern "C" int nh_bench_probe_pattern(nh_db *db, int lanes, int depth, int blocks_per_sm, double p_continue,
                                      uint64_t sm_window_bytes, uint32_t items_per_chain, int iters,
                                      double *out_items_per_s, double *out_requests_per_s) {
  if (!db || !out_items_per_s || !out_requests_per_s || iters < 1 || items_per_chain < 1 ||
      (lanes != 0 && lanes != 1 && lanes != 2 && lanes != 4) || (depth != 1 && depth != 2 && depth != 4) ||
      (lanes == 0 && (depth == 4 || sm_window_bytes)) || blocks_per_sm < 1 ||
      blocks_per_sm > 8 || !(p_continue >= 0.0 && p_continue < 1.0))
    return nh_set_error(NH_ERR_INVALID, "bad argument");
  CUDA_TRY(cudaSetDevice(db->info.device));
  const uint64_t n_sectors = db->info.capacity / 8;
  if (n_sectors < 64 || (sm_window_bytes && sm_window_bytes / 32 > n_sectors))
    return nh_set_error(NH_ERR_INVALID, "table too small");
  uint32_t *sink = nullptr;
  unsigned long long *d_cnt = nullptr;
  CUDA_TRY(cudaMalloc(&sink, 64));
  CUDA_TRY(cudaMalloc(&d_cnt, 16));
  cudaStream_t st;
  CUDA_TRY(cudaStreamCreate(&st));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0);
  cudaEventCreate(&e1);
  const uint32_t p_thresh = (uint32_t)(p_continue * 4294967296.0);
  double best_items = 0, best_req = 0;
  for (int i = 0; i < iters + 1; i++) { /* first launch is warm-up */
    cudaMemsetAsync(d_cnt, 0, 16, st);
    cudaEventRecord(e0, st);
    nh_launch_probe_pattern(db->d_cells, n_sectors, lanes, depth, blocks_per_sm, items_per_chain, p_thresh,
                            0x1234567ULL * (uint64_t)(i + 1), sm_window_bytes / 32, d_cnt, sink, db->sm_count, st);
    cudaEventRecord(e1, st);
    unsigned long long h[2] = {0, 0};
    cudaMemcpyAsync(h, d_cnt, 16, cudaMemcpyDeviceToHost, st);
    cudaStreamSynchronize(st);
    float ms = 0;
    cudaEventElapsedTime(&ms, e0, e1);
    if (i > 0 && ms > 0 && (double)h[0] / ms > best_items) {
      best_items = (double)h[0] / ms;
      best_req = (double)h[1] / ms;
    }
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaStreamDestroy(st);
  cudaFree(sink);
  cudaFree(d_cnt);
  CUDA_TRY(cudaGetLastError());
  *out_items_per_s = best_items * 1e3;
  *out_requests_per_s = best_req * 1e3;
  return NH_OK;
}

/* the p = 0 case of the pattern above, in GB/s of 32-byte sectors (kept for callers of ABI 1) */
extern "C" int nh_bench_random_gather(nh_db *db, uint64_t n_reads, int iters, double *out_gbs) {
  if (!db || !out_gbs || iters < 1) return nh_set_error(NH_ERR_INVALID, "bad argument");
  const uint64_t chains = (uint64_t)db->sm_count * 8 * 256 * 4;
  uint64_t per = n_reads / chains;
  if (per < 1) per = 1;
  double items = 0, req = 0;
  int rc = nh_bench_probe_pattern(db, 1, 4, 8, 0.0, 0, (uint32_t)per, iters, &items, &req);
  if (rc) return rc;
  *out_gbs = req * 32.0 / 1e9;
  return NH_OK;
}
