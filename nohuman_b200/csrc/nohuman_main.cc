/*
 * nohuman_main.cc — command-line front end over libnohuman_gpu.so with the
 * flag surface of the reference CLI (mbhall88/nohuman src/main.rs:21-104) for
 * the path this repository rebuilds: --db / NOHUMAN_DB / --db-version, --conf,
 * -t, one or two inputs, --out1/--out2, -F, -H.  The external kraken2 process
 * (src/main.rs:170-270) and the compression pass after it (src/main.rs:340-368)
 * are one call to nh_run_files().  --list-db-versions reads the manifest the way
 * download_config does when a local config.toml exists (src/download.rs:146-168,
 * config.toml:1-19); its network half and --download are not reproduced
 * (SURVEY.md §2 row 10).
 *
 * The same binary installed under the name `kraken2` accepts the argv nohuman
 * builds (src/main.rs:215-267) and prints the three stderr lines
 * parse_kraken_stderr reads (src/lib.rs:61-97), so an unmodified nohuman can
 * run on the GPU by putting it first on $PATH.
 */
#include <getopt.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/stat.h>
#include <time.h>

#include <algorithm>
#include <charconv>
#include <string>
#include <vector>

#include <dirent.h>

#include "../../include/nohuman_gpu.h"

static bool g_verbose = false;

static void logmsg(const char *level, const char *fmt, ...) {
  if (!strcmp(level, "DEBUG") && !g_verbose) return;
  char ts[32];
  time_t t = time(nullptr);
  struct tm tmv;
  gmtime_r(&t, &tmv);
  strftime(ts, sizeof ts, "%Y-%m-%dT%H:%M:%SZ", &tmv);
  fprintf(stderr, "[%s %-5s] ", ts, level);
  va_list ap;
  va_start(ap, fmt);
  vfprintf(stderr, fmt, ap);
  va_end(ap);
  fputc('\n', stderr);
}

static bool is_dir(const std::string &p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}
static bool exists(const std::string &p) {
  struct stat st;
  return stat(p.c_str(), &st) == 0;
}

/* ---- std::path helpers with Rust's Path semantics (src/main.rs:274-307) ---- */
static std::string path_parent(const std::string &p) {
  size_t s = p.find_last_of('/');
  if (s == std::string::npos) return "";
  return s == 0 ? "/" : p.substr(0, s);
}
static std::string path_file_name(const std::string &p) {
  size_t s = p.find_last_of('/');
  return s == std::string::npos ? p : p.substr(s + 1);
}
/* Path::extension: text after the last '.', none if the name starts with its only dot */
static bool path_extension(const std::string &p, std::string &ext) {
  std::string f = path_file_name(p);
  size_t d = f.find_last_of('.');
  if (d == std::string::npos || d == 0) return false;
  ext = f.substr(d + 1);
  return true;
}
static std::string path_file_stem(const std::string &p) {
  std::string f = path_file_name(p);
  size_t d = f.find_last_of('.');
  if (d == std::string::npos || d == 0) return f;
  return f.substr(0, d);
}
static std::string path_join(const std::string &a, const std::string &b) {
  if (a.empty()) return b;
  return a.back() == '/' ? a + b : a + "/" + b;
}

/* ---- CompressionFormat (src/compression.rs:11-118, 271-296) ---- */
static const char *format_ext(int f) {
  switch (f) {
    case 'b': return "bz2";
    case 'g': return "gz";
    case 'x': return "xz";
    case 'z': return "zst";
    default: return "";
  }
}
static int format_from_path(const std::string &p) {
  std::string e;
  if (!path_extension(p, e)) return 'u';
  if (e == "bz2") return 'b';
  if (e == "gz") return 'g';
  if (e == "xz") return 'x';
  if (e == "zst" || e == "zstd") return 'z';
  return 'u';
}
static bool format_from_magic(const std::string &p, int *fmt, std::string &err) {
  FILE *f = fopen(p.c_str(), "rb");
  unsigned char m[5];
  if (!f || fread(m, 1, 5, f) != 5) {
    if (f) fclose(f);
    err = "Failed to read the first five bytes of the file";
    return false;
  }
  fclose(f);
  if (m[0] == 0x1f && m[1] == 0x8b)
    *fmt = 'g';
  else if (m[0] == 0x42 && m[1] == 0x5a)
    *fmt = 'b';
  else if (m[0] == 0x28 && m[1] == 0xb5 && m[2] == 0x2f && m[3] == 0xfd)
    *fmt = 'z';
  else if (m[0] == 0xfd && m[1] == 0x37 && m[2] == 0x7a && m[3] == 0x58 && m[4] == 0x5a)
    *fmt = 'x';
  else
    *fmt = 'u';
  return true;
}
static std::string add_extension(int fmt, const std::string &p) {
  if (fmt == 'u') return p;
  return p + "." + format_ext(fmt); /* "<ext>.<new>" when an extension exists, else ".<new>" */
}
/* default output name: <dir>/<stem>.nohuman.fq[.ext] (src/main.rs:274-290) */
static std::string default_output(const std::string &input, int out_fmt) {
  std::string ext = format_ext(format_from_path(input));
  std::string cur;
  bool has = path_extension(input, cur);
  std::string stem;
  if ((has ? cur : std::string()) == ext) {
    std::string no_ext = has ? path_join(path_parent(input), path_file_stem(input)) : input;
    stem = path_file_stem(no_ext);
  } else {
    stem = path_file_stem(input);
  }
  return add_extension(out_fmt, path_join(path_parent(input), stem + ".nohuman.fq"));
}

/* ---- database resolution (src/lib.rs:119-141, src/main.rs:393-434, src/download.rs:178-234) ---- */
static bool validate_db_directory(const std::string &p, std::string &out) {
  const char *req[3] = {"hash.k2d", "opts.k2d", "taxo.k2d"};
  for (const std::string &c : {p, path_join(p, "db")}) {
    bool all = is_dir(c);
    for (auto r : req) all = all && exists(path_join(c, r));
    if (all) {
      out = c;
      return true;
    }
  }
  return false;
}
struct Installed {
  std::string version, path, added;
};
/* nohuman-db.toml: version = "..." / added = "YYYY-MM-DD" */
static bool read_metadata(const std::string &dir, Installed &out) {
  FILE *f = fopen(path_join(dir, "nohuman-db.toml").c_str(), "r");
  if (!f) return false;
  char line[512];
  bool v = false, a = false;
  while (fgets(line, sizeof line, f)) {
    char key[64], val[256];
    if (sscanf(line, " %63[a-z_] = \"%255[^\"]\"", key, val) == 2) {
      if (!strcmp(key, "version")) out.version = val, v = true;
      if (!strcmp(key, "added")) out.added = val, a = true;
    }
  }
  fclose(f);
  return v && a;
}
static bool valid_date(const std::string &s) {
  int y, m, d;
  char tail;
  return sscanf(s.c_str(), "%4d-%2d-%2d%c", &y, &m, &d, &tail) == 3 && m >= 1 && m <= 12 && d >= 1 && d <= 31;
}
/* ---- database manifest (config.toml; src/download.rs:54-98,146-176) ---- */
struct Release {
  std::string version, url, md5, added;
};
struct Manifest {
  std::string default_version;
  std::vector<Release> databases;
};
/* The subset of TOML the manifest uses: `key = "value"` lines and `[[databases]]` table headers.
 * Returns an error text (empty on success); like the reference every `added` must be a date. */
static std::string read_manifest(const std::string &path, Manifest &out) {
  FILE *f = fopen(path.c_str(), "r");
  if (!f) return "Failed to download database config"; /* DownloadError::ConfigDownloadFailed: no local file, no network */
  char line[1024];
  Release *cur = nullptr;
  bool ok = true;
  while (fgets(line, sizeof line, f)) {
    char *p = line;
    while (*p == ' ' || *p == '\t') p++;
    if (*p == '#' || *p == '\n' || *p == '\r' || !*p) continue;
    if (!strncmp(p, "[[databases]]", 13)) {
      out.databases.emplace_back();
      cur = &out.databases.back();
      continue;
    }
    if (*p == '[') { /* some other table: not ours */
      cur = nullptr;
      continue;
    }
    char key[64], val[512];
    if (sscanf(p, "%63[A-Za-z0-9_-] = \"%511[^\"]\"", key, val) != 2) {
      ok = false;
      continue;
    }
    if (!cur) {
      if (!strcmp(key, "default_version")) out.default_version = val;
    } else if (!strcmp(key, "version")) cur->version = val;
    else if (!strcmp(key, "url")) cur->url = val;
    else if (!strcmp(key, "md5")) cur->md5 = val;
    else if (!strcmp(key, "added")) cur->added = val;
  }
  fclose(f);
  for (auto &r : out.databases)
    if (r.version.empty() || r.url.empty() || r.md5.empty() || r.added.empty()) ok = false;
  if (!ok) return "Failed to parse database config";
  for (auto &r : out.databases)
    if (!valid_date(r.added)) return "Invalid date '" + r.added + "' in database manifest";
  return "";
}

static std::vector<Installed> installed_databases(const std::string &root) {
  std::vector<Installed> v;
  if (DIR *d = opendir(root.c_str())) {
    while (struct dirent *e = readdir(d)) {
      if (e->d_name[0] == '.') continue;
      std::string p = path_join(root, e->d_name), actual;
      Installed ins;
      if (is_dir(p) && read_metadata(p, ins) && validate_db_directory(p, actual)) {
        ins.path = p;
        v.push_back(ins);
      }
    }
    closedir(d);
  }
  std::string actual;
  Installed tmp;
  if (validate_db_directory(root, actual) && !read_metadata(root, tmp)) v.push_back({"legacy", root, "1970-01-01"});
  return v;
}

/* ---- confidence: f32, then the shortest decimal re-read as a double (src/main.rs:213) ---- */
static bool parse_confidence(const char *s, double *out, std::string &err) {
  char *end = nullptr;
  float f = strtof(s, &end);
  if (end == s || *end) {
    err = "Confidence score must be a number";
    return false;
  }
  if (!(f >= 0.0f && f <= 1.0f)) {
    err = "Confidence score must be in the closed interval [0, 1]";
    return false;
  }
  char buf[64];
  auto r = std::to_chars(buf, buf + sizeof buf - 1, f); /* shortest round-trip, as Rust's Display */
  *r.ptr = 0;
  *out = strtod(buf, nullptr);
  return true;
}

static int fail(const char *fmt, ...) {
  fprintf(stderr, "Error: ");
  va_list ap;
  va_start(ap, fmt);
  vfprintf(stderr, fmt, ap);
  va_end(ap);
  fputc('\n', stderr);
  return 1;
}

static double pct(uint64_t a, uint64_t b) { return b ? 100.0 * (double)a / (double)b : 0.0 / 0.0; }

/* ------------------------------------------------------------------ */
/* invoked as `kraken2`: the argv of src/main.rs:215-267                */

static int kraken2_shim(int argc, char **argv) {
  static option opts[] = {{"threads", 1, 0, 't'},        {"db", 1, 0, 'd'},           {"output", 1, 0, 'o'},
                          {"confidence", 1, 0, 'c'},     {"report", 1, 0, 'r'},       {"paired", 0, 0, 'p'},
                          {"classified-out", 1, 0, 'C'}, {"unclassified-out", 1, 0, 'U'}, {"version", 0, 0, 'V'},
                          {0, 0, 0, 0}};
  int threads = 1, paired = 0;
  std::string db, output, report, cls_out, uncls_out;
  double conf = 0.0;
  int c;
  while ((c = getopt_long(argc, argv, "", opts, nullptr)) != -1) switch (c) {
      case 't': threads = atoi(optarg); break;
      case 'd': db = optarg; break;
      case 'o': output = optarg; break;
      case 'c': conf = strtod(optarg, nullptr); break; /* kraken2 reads a double */
      case 'r': report = optarg; break;
      case 'p': paired = 1; break;
      case 'C': cls_out = optarg; break;
      case 'U': uncls_out = optarg; break;
      case 'V': printf("Kraken version 2.17 (libnohuman_gpu, ABI %d)\n", nh_abi_version()); return 0;
      default: return 64;
    }
  std::vector<std::string> in(argv + optind, argv + argc);
  if (db.empty() || in.empty() || in.size() > 2 || (paired && in.size() != 2)) {
    fprintf(stderr, "kraken2 (GPU shim): need --db and one input file (two with --paired)\n");
    return 64;
  }
  if (cls_out.empty() == uncls_out.empty()) {
    fprintf(stderr, "kraken2 (GPU shim): exactly one of --classified-out / --unclassified-out is supported\n");
    return 64;
  }
  std::string tmpl = cls_out.empty() ? uncls_out : cls_out, o1 = tmpl, o2;
  if (paired) {
    size_t h = tmpl.find('#');
    if (h == std::string::npos) {
      fprintf(stderr, "Paired filename format missing # character: %s\n", tmpl.c_str());
      return 64;
    }
    o1 = tmpl.substr(0, h) + "_1" + tmpl.substr(h + 1);
    o2 = tmpl.substr(0, h) + "_2" + tmpl.substr(h + 1);
  }
  nh_db *dbh = nullptr;
  nh_session *sess = nullptr;
  nh_params_t p;
  memset(&p, 0, sizeof p);
  p.confidence = conf;
  p.minimum_hit_groups = -1;
  p.paired = paired;
  p.keep_human = !cls_out.empty();
  p.threads = threads;
  p.max_batch_bases = 1u << 20; /* parameter carrier only: nh_run_files sizes its own sessions per chunk */
  p.max_batch_seqs = 1u << 12;
  nh_files_t f;
  memset(&f, 0, sizeof f);
  f.in1 = in[0].c_str();
  f.in2 = paired ? in[1].c_str() : nullptr;
  f.out1 = o1.c_str();
  f.out2 = paired ? o2.c_str() : nullptr;
  f.out_format = 'u';
  f.tag_classified = 1;
  f.kraken_output = output.empty() || output == "-" ? nullptr : output.c_str();
  f.kraken_report = report.empty() ? nullptr : report.c_str();
  nh_run_stats_t st;
  memset(&st, 0, sizeof st);
  if (nh_db_open(db.c_str(), 0, &dbh) || nh_session_create(dbh, &p, &sess) || nh_run_files(sess, &f, &st)) {
    fprintf(stderr, "classify: %s\n", nh_last_error());
    return 1;
  }
  nh_session_destroy(sess);
  nh_db_close(dbh);
  const double mbp = st.bases / 1e6, secs = st.seconds > 0 ? st.seconds : 1e-9;
  fprintf(stderr, "%llu sequences (%.2f Mbp) processed in %.3fs (%.1f Kseq/m, %.2f Mbp/m).\n",
          (unsigned long long)st.total, mbp, secs, st.total / 1e3 / (secs / 60), mbp / (secs / 60));
  fprintf(stderr, "  %llu sequences classified (%.2f%%)\n", (unsigned long long)st.classified, pct(st.classified, st.total));
  fprintf(stderr, "  %llu sequences unclassified (%.2f%%)\n", (unsigned long long)st.unclassified,
          pct(st.unclassified, st.total));
  return 0;
}

/* ------------------------------------------------------------------ */

static void usage() {
  puts("Remove human reads from a sequencing run (B200 build of nohuman's kraken2 path)\n\n"
       "Usage: nohuman [OPTIONS] [INPUT]...\n\n"
       "Arguments:\n  [INPUT]...  Input file(s) to remove human reads from\n\n"
       "Options:\n"
       "  -o, --out1 <OUTPUT_1>      First output file [default: <input_1 stem>.nohuman.fq(.ext)]\n"
       "  -O, --out2 <OUTPUT_2>      Second output file\n"
       "  -c, --check                Check that all required dependencies are available and exit\n"
       "  -D, --db <PATH>            Path to the database [env: NOHUMAN_DB] [default: ~/.nohuman/db]\n"
       "      --db-version <VERSION> Name of the installed database version to use (defaults to the newest installed)\n"
       "  -F, --output-type <FORMAT> Output compression format. u: uncompressed; b: Bzip2; g: Gzip; x: Xz (Lzma); z: Zstd\n"
       "  -t, --threads <INT>        Number of host threads (parsing, output compression). Cannot be 0 [default: 1]\n"
       "  -H, --human                Output human reads instead of removing them\n"
       "  -C, --conf <[0, 1]>        Kraken2 minimum confidence score [default: 0.0]\n"
       "  -k, --kraken-output <FILE> Write the Kraken2 read classification output to a file\n"
       "  -r, --kraken-report <FILE> Write the Kraken2 report with aggregate counts/clade to file\n"
       "      --gpu <ID>             First CUDA device to use [default: 0]\n"
       "      --gpus <N|all>         Number of GPUs: read batches are sharded, the database is replicated [default: 1]\n"
       "      --gpu-gzip             Compress gzip output (-F g) on the GPUs instead of the host threads\n"
       "  -v, --verbose              Set the logging level to verbose\n"
       "  -h, --help                 Print help\n"
       "  -V, --version              Print version");
}

int main(int argc, char **argv) {
  if (path_file_name(argv[0]) == "kraken2") return kraken2_shim(argc, argv);
  static option opts[] = {{"out1", 1, 0, 'o'},         {"out2", 1, 0, 'O'},          {"check", 0, 0, 'c'},
                          {"download", 0, 0, 'd'},     {"db", 1, 0, 'D'},            {"db-version", 1, 0, 1},
                          {"list-db-versions", 0, 0, 2}, {"output-type", 1, 0, 'F'}, {"threads", 1, 0, 't'},
                          {"human", 0, 0, 'H'},        {"conf", 1, 0, 'C'},          {"kraken-output", 1, 0, 'k'},
                          {"kraken-report", 1, 0, 'r'}, {"verbose", 0, 0, 'v'},      {"help", 0, 0, 'h'},
                          {"version", 0, 0, 'V'},      {"gpu", 1, 0, 3},             {"plan", 0, 0, 4},
                          {"gpus", 1, 0, 5},           {"gpu-gzip", 0, 0, 6},
                          {0, 0, 0, 0}};
  std::string out1, out2, db, db_version, kraken_output, kraken_report, err;
  bool check = false, download = false, list = false, human = false, plan = false, gpu_gzip = false;
  int out_type = 0, gpu = 0, gpus = 1;
  long threads = 1;
  double conf = 0.0;
  if (const char *e = getenv("NOHUMAN_DB")) db = e;
  int c;
  while ((c = getopt_long(argc, argv, "o:O:cdD:F:t:HC:k:r:vhV", opts, nullptr)) != -1) switch (c) {
      case 'o': out1 = optarg; break;
      case 'O': out2 = optarg; break;
      case 'c': check = true; break;
      case 'd': download = true; break;
      case 'D': db = optarg; break;
      case 1: db_version = optarg; break;
      case 2: list = true; break;
      case 'F': {
        std::string s = optarg;
        std::transform(s.begin(), s.end(), s.begin(), ::tolower);
        if (s.size() != 1 || !strchr("bgxzu", s[0])) return fail("Invalid compression format: %s", optarg);
        out_type = s[0];
        break;
      }
      case 't':
        threads = strtol(optarg, nullptr, 10);
        if (threads < 1) return fail("invalid value '%s' for '--threads <INT>': number would be zero for non-zero type", optarg);
        break;
      case 'H': human = true; break;
      case 'C':
        if (!parse_confidence(optarg, &conf, err)) return fail("invalid value '%s' for '--conf <[0, 1]>': %s", optarg, err.c_str());
        break;
      case 'k': kraken_output = optarg; break;
      case 'r': kraken_report = optarg; break;
      case 'v': g_verbose = true; break;
      case 'h': usage(); return 0;
      case 'V': printf("nohuman 0.5.1 (B200 hot path, libnohuman_gpu ABI %d)\n", nh_abi_version()); return 0;
      case 3: gpu = atoi(optarg); break;
      case 5: gpus = !strcmp(optarg, "all") ? -1 : atoi(optarg); break;
      case 4: plan = true; break; /* hidden: print what would run (database, format, outputs) and exit */
      case 6: gpu_gzip = true; break;
      default: return 2;
    }
  std::vector<std::string> input(argv + optind, argv + argc);
  for (auto &p : input)
    if (!exists(p)) return fail("invalid value '%s' for '[INPUT]...': \"%s\" does not exist", p.c_str(), p.c_str());
  if (db.empty()) {
    const char *home = getenv("HOME");
    db = path_join(path_join(home ? home : "", ".nohuman"), "db");
  }
  if (list) {
    /* src/main.rs:123-147 over download_config (src/download.rs:146-168): ./config.toml first; the
     * reference would fetch CONFIG_URL next, which this build does not do */
    Manifest m;
    const std::string err = read_manifest("config.toml", m);
    if (!err.empty())
      return fail("Failed to download database manifest: %s%s", err.c_str(),
                  exists("config.toml") ? "" : " (no config.toml in the working directory; this build does not fetch it from the network)");
    printf("Available databases:\n");
    for (auto &r : m.databases)
      printf("- %s%s (added %s) -> %s\n", r.version.c_str(), r.version == m.default_version ? " (default)" : "",
             r.added.c_str(), r.url.c_str());
    return 0;
  }
  if (download)
    return fail("--download needs network access, which this build does not include; "
                "install a database directory (hash.k2d, opts.k2d, taxo.k2d) and pass it with --db");
  if (!plan && nh_device_count() < 1) {
    logmsg("ERROR", "The following dependencies are missing:");
    logmsg("ERROR", "a CUDA device (libnohuman_gpu has no CPU path)");
    return fail("Missing dependencies");
  }
  if (check) {
    logmsg("INFO", "All dependencies are available");
    return 0;
  }
  if (input.empty()) return fail("No input files provided");
  if (input.size() > 2) return fail("Only one or two input files are allowed");

  /* resolve_database (src/main.rs:393-434) */
  std::string db_path, version;
  if (!db_version.empty()) {
    if (db_version == "all")
      return fail("Cannot run with `--db-version all`. Use `--download --db-version all` to download every database.");
    bool found = false;
    for (auto &i : installed_databases(db))
      if (i.version == db_version) {
        found = validate_db_directory(i.path, db_path);
        version = i.version;
        break;
      }
    if (!found)
      return fail("Database version '%s' is not installed under \"%s\". Run `nohuman --download --db-version %s` to download it.",
                  db_version.c_str(), db.c_str(), db_version.c_str());
  } else if (!validate_db_directory(db, db_path)) {
    std::vector<Installed> all = installed_databases(db);
    if (all.empty()) return fail("Database does not exist at \"%s\". Run `nohuman --download` to fetch one.", db.c_str());
    auto key = [](const Installed &i) { return valid_date(i.added) ? i.added : std::string("1970-01-01"); };
    const Installed *best = &all[0];
    for (auto &i : all)
      if (key(i) >= key(*best)) best = &i;
    validate_db_directory(best->path, db_path);
    version = best->version;
  }
  if (!version.empty())
    logmsg("INFO", "Using database version %s at \"%s\"", version.c_str(), db_path.c_str());
  else
    logmsg("INFO", "Using database at \"%s\"", db_path.c_str());

  /* output format: -F, else extension of --out1, else magic bytes of the first input (src/main.rs:238-245) */
  int fmt = out_type;
  if (!fmt) {
    if (!out1.empty())
      fmt = format_from_path(out1);
    else if (!format_from_magic(input[0], &fmt, err))
      return fail("%s", err.c_str());
  }
  const bool paired = input.size() == 2;
  if (out1.empty()) out1 = default_output(input[0], fmt);
  if (paired && out2.empty()) out2 = default_output(input[1], fmt);

  if (plan) {
    printf("db=%s\nversion=%s\nformat=%c\nout1=%s\nout2=%s\npaired=%d\nkeep_human=%d\nconfidence=%.17g\nthreads=%ld\n"
           "gpu_gzip=%d\n",
           db_path.c_str(), version.c_str(), fmt, out1.c_str(), out2.c_str(), (int)paired, (int)human, conf, threads,
           (int)gpu_gzip);
    return 0;
  }
  /* more GPUs: the table is read from disk once and broadcast (NCCL over NVLink, else peer copies);
   * nothing is exchanged between the GPUs afterwards */
  if (gpus < 0) gpus = nh_device_count() - gpu;
  if (gpus < 1 || gpu + gpus > nh_device_count()) return fail("--gpus %d from device %d: only %d device(s) visible", gpus, gpu, nh_device_count());
  std::vector<int> devs;
  for (int g = 0; g < gpus; g++) devs.push_back(gpu + g);
  std::vector<nh_db *> replicas((size_t)gpus, nullptr);
  struct timespec t_load0, t_load1;
  clock_gettime(CLOCK_MONOTONIC, &t_load0);
  if (nh_db_open_multi(db_path.c_str(), devs.data(), gpus, replicas.data())) return fail("%s", nh_last_error());
  clock_gettime(CLOCK_MONOTONIC, &t_load1);
  nh_params_t p;
  memset(&p, 0, sizeof p);
  p.confidence = conf;
  p.minimum_hit_groups = -1;
  p.paired = paired;
  p.keep_human = human;
  p.threads = (int)threads;
  p.gpu_gzip = gpu_gzip;
  p.max_batch_bases = 1u << 20; /* parameter carrier only: nh_run_files sizes its own sessions */
  p.max_batch_seqs = 1u << 12;
  std::vector<nh_session *> sessions;
  for (int g = 0; g < gpus; g++) {
    nh_session *rs = nullptr;
    if (nh_session_create(replicas[(size_t)g], &p, &rs)) return fail("%s", nh_last_error());
    sessions.push_back(rs);
  }
  {
    nh_db_info_t di;
    memset(&di, 0, sizeof di);
    if (gpus > 1) nh_db_info(replicas[1], &di);
    const double load_s = (double)(t_load1.tv_sec - t_load0.tv_sec) + 1e-9 * (double)(t_load1.tv_nsec - t_load0.tv_nsec);
    if (gpus > 1)
      logmsg("INFO", "Database replicated on %d GPUs (%s)", gpus, di.replicated_by == 1 ? "NCCL broadcast" : "peer copies");
    logmsg("DEBUG", "database load: %.3f s on %d GPU(s)", load_s, gpus);
  }
  logmsg("INFO", human ? "Keeping human reads..." : "Removing human reads...");
  nh_files_t f;
  memset(&f, 0, sizeof f);
  f.in1 = input[0].c_str();
  f.in2 = paired ? input[1].c_str() : nullptr;
  f.out1 = out1.c_str();
  f.out2 = paired ? out2.c_str() : nullptr;
  f.out_format = fmt;
  f.tag_classified = 1;
  f.kraken_output = kraken_output.empty() ? nullptr : kraken_output.c_str();
  f.kraken_report = kraken_report.empty() ? nullptr : kraken_report.c_str();
  nh_run_stats_t st;
  memset(&st, 0, sizeof st);
  if (nh_run_files_multi(sessions.data(), (int)sessions.size(), &f, &st)) return fail("Failed to run kraken2: %s", nh_last_error());
  /* the line CommandRunner::run logs from kraken2's stderr (src/lib.rs:38-45) */
  logmsg("INFO", "%llu / %llu (%.2f%%) sequences classified as human; %llu (%.2f%%) as non-human",
         (unsigned long long)st.classified, (unsigned long long)st.total, pct(st.classified, st.total),
         (unsigned long long)st.unclassified, pct(st.unclassified, st.total));
  logmsg("INFO", "Kraken2 finished. Organising output...");
  logmsg("INFO", "Output file written to: \"%s\"", out1.c_str());
  if (paired) logmsg("INFO", "Output file written to: \"%s\"", out2.c_str());
  logmsg("DEBUG", "%.3f s, %.2f Mbp", st.seconds, st.bases / 1e6);
  logmsg("DEBUG", "busy seconds per stage (summed over its threads): inflate %.2f (%d thr), parse %.2f, stage %.2f, classify %.2f, "
                  "serialise %.2f, compress %.2f (%d thr), write %.2f",
         st.busy_inflate_s, st.threads_inflate, st.busy_parse_s, st.busy_stage_s, st.busy_classify_s, st.busy_serialise_s,
         st.busy_compress_s, st.threads_compress, st.busy_write_s);
  for (auto *x : sessions) nh_session_destroy(x);
  for (auto *x : replicas) nh_db_close(x);
  logmsg("INFO", "Done.");
  return 0;
}
