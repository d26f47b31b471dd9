// main.cpp -- `raxtax` command-line binary on top of the B200 library (SURVEY.md 8(f) rows 1, 3, 4).
//
// Mirrors the reference's CLI surface, output files and restart behaviour (src/io.rs:112-300, src/main.rs:14-173):
//   raxtax -d <db.fasta[.gz] | db.bin> -i <queries.fasta[.gz]> [-o PREFIX] [--skip-exact-matches] [--raw-confidence] [--tsv]
//          [--redo] [--only-db] [--skip-db] [-c] [-t N] [--pin] [-v|-q] [--gpu N] [--gpus N [--shard-references]] [--batch N]
//          [--strand plus|both] [--best-hits N]
// writes <PREFIX>/raxtax.out, raxtax.log, raxtax.ckp, raxtax.json, (with --tsv) raxtax.tsv in the reference's formats and (with
// --best-hits) raxtax.hits, each query's N references with the most shared 8-mers
// (lineage.rs:17-48), and <PREFIX>/<database stem>.bin, the bincode database of tree.rs:146-164, unless --skip-db.
// A database path that deserialises as such a .bin is loaded instead of parsed (parser.rs:37-44).  An interrupted run is
// continued from raxtax.json + raxtax.ckp (io.rs:47-90,156-230) when the flags and the database fingerprint still match.
// One deliberate difference: --clean removes the checkpoint files and a database this run family created under PREFIX,
// never the file the user passed with -d (Checkpoint::cleanup, io.rs:80-89, would delete it when --skip-db was given).
// Not carried over: thread pinning (accepted, no effect: the hot path runs on the GPU).
// Exit codes follow main.rs: 73 CANTCREAT, 66 NOINPUT, 74 IOERR, 75 TEMPFAIL, 0 OK.

#include <sys/stat.h>

#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <fstream>
#include <set>
#include <sstream>
#include <string>
#include <vector>

#include "raxtax_host.h"

namespace {

enum { EX_OK_ = 0, EX_USAGE_ = 64, EX_NOINPUT_ = 66, EX_CANTCREAT_ = 73, EX_IOERR_ = 74, EX_TEMPFAIL_ = 75 };

struct Args {
    std::string database_path, query_file, prefix = "raxtax";
    bool skip_exact_matches = false, tsv = false, only_db = false, skip_db = false, clean = false, raw_confidence = false, redo = false,
         pin = false, shard_refs = false, both_strands = false;
    int threads = 0, verbosity = 3 /* Info */, gpu = 0, gpus = 1;
    unsigned best_hits = 0;  // --best-hits: 0 = no raxtax.hits
    size_t batch = 0;
};

void usage() {
    fprintf(stderr,
            "Usage: raxtax [OPTIONS] --database-path <DATABASE_PATH>\n\n"
            "Options:\n"
            "  -d, --database-path <DATABASE_PATH>  Path to the database fasta or bin file (.gz/.gzip fasta accepted)\n"
            "  -i, --query-file <QUERY_FILE>        Path to the query file\n"
            "      --skip-exact-matches             If used for mislabling analysis, you want to skip exact sequence matches\n"
            "      --tsv                            Output primary result file in tsv format\n"
            "      --only-db                        Only create the binary database and exit\n"
            "      --skip-db                        Don't create the binary database\n"
            "  -c, --clean                          Remove checkpoint files after a successful run\n"
            "      --raw-confidence                 Don't adjust confidence values for 1 exact match\n"
            "  -t, --threads <THREADS>              Accepted for compatibility (the hot path runs on the GPU)\n"
            "  -o, --prefix <PREFIX>                Output prefix [default: raxtax]\n"
            "      --redo                           Force override of existing output files\n"
            "      --pin                            Accepted for compatibility\n"
            "      --gpu <ORDINAL>                  First CUDA device to use [default: 0]\n"
            "      --gpus <N>                       Number of GPUs (ORDINAL .. ORDINAL+N-1): queries are partitioned, the index is\n"
            "                                       replicated [default: 1]\n"
            "      --shard-references               With --gpus N: every GPU holds 1/N of the references (databases too large to\n"
            "                                       replicate) instead of the whole index\n"
            "      --batch <N>                      Queries per device batch [default: all]\n"
            "      --strand <STRAND>                plus: classify the queries as given; both: in the orientation that shares more\n"
            "                                       8-mers with some reference, strand column +/- in the outputs [default: plus]\n"
            "      --best-hits <N>                  Write each query's N (1..64) references with the most shared 8-mers to\n"
            "                                       raxtax.hits: label, rank, lineage, shared 8-mers, K, reference id\n"
            "  -v, --verbose...                     Increase logging verbosity (repeatable: -vv)\n"
            "  -q, --quiet...                       Decrease logging verbosity (repeatable: -qq)\n");
}

struct Writers {
    FILE *primary = nullptr, *tsv = nullptr, *log = nullptr, *progress = nullptr, *hits = nullptr;
    int verbosity = 3;
    std::string pending_labels;  // labels whose result lines are written but possibly still in a stdio buffer
    size_t pending_n = 0;
    bool failed = false;

    // The reference writes unbuffered Files in the order result, then progress (main.rs:128-134): the progress file can never run
    // ahead of the output.  Here the streams are block-buffered, so the labels are held back until the result lines they stand for
    // have been flushed; a kill at any point leaves raxtax.ckp listing only queries whose lines are complete in raxtax.out / .tsv
    // (lines of queries not yet listed are what check_incomplete_output removes on resume).
    bool commit() {
        if (pending_n == 0) return !failed;
        if ((tsv && fflush(tsv) != 0) || (hits && fflush(hits) != 0) || fflush(primary) != 0) failed = true;
        if (!failed && (fwrite(pending_labels.data(), 1, pending_labels.size(), progress) != pending_labels.size() || fflush(progress) != 0)) failed = true;
        pending_labels.clear();
        pending_n = 0;
        return !failed;
    }
};

int send_cb(void* user, const char* label, const char* primary, const char* tsv) {  // writer thread body (main.rs:128-134)
    Writers* w = (Writers*)user;
    if (w->tsv && tsv && (fputs(tsv, w->tsv) < 0 || fputc('\n', w->tsv) == EOF)) return 1;
    if (fputs(primary, w->primary) < 0 || fputc('\n', w->primary) == EOF) return 1;
    w->pending_labels += label;
    w->pending_labels += '\n';
    if (++w->pending_n >= 256 && !w->commit()) return 1;
    return 0;
}

int hits_cb(void* user, const char* /*label*/, const char* lines) {  // called right before send_cb of the same query
    Writers* w = (Writers*)user;
    if (*lines && (fputs(lines, w->hits) < 0 || fputc('\n', w->hits) == EOF)) return 1;
    return 0;
}

void log_cb(void* user, int level, const char* msg) {  // env_logger without timestamps/targets (main.rs:34-39)
    Writers* w = (Writers*)user;
    if (level > w->verbosity) return;
    fprintf(w->log, "[%s] %s\n", level == 2 ? "WARN " : "INFO ", msg);
}

bool exists(const std::string& p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0;
}
bool is_file(const std::string& p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISREG(st.st_mode);
}
bool is_dir(const std::string& p) {
    struct stat st;
    return stat(p.c_str(), &st) == 0 && S_ISDIR(st.st_mode);
}
// std::path::absolute (Unix): the path joined onto the working directory when relative, `.` components and repeated separators
// dropped, `..` KEPT, no symlink resolution, no existence check -- the string raxtax.json's fingerprint compares (io.rs:23-45)
std::string absolute(const std::string& p) {
    std::string full = p;
    if (p.empty() || p[0] != '/') {
        std::error_code ec;
        const auto cwd = std::filesystem::current_path(ec);
        if (ec) return p;
        full = cwd.string() + "/" + p;
    }
    std::string out;
    size_t i = 0;
    while (i < full.size()) {
        while (i < full.size() && full[i] == '/') ++i;
        size_t j = i;
        while (j < full.size() && full[j] != '/') ++j;
        if (j > i && !(j - i == 1 && full[i] == '.')) {
            out += '/';
            out.append(full, i, j - i);
        }
        i = j;
    }
    return out.empty() ? "/" : out;
}
bool read_raw(const std::string& path, std::string* out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    char buf[1 << 16];
    size_t n;
    while ((n = fread(buf, 1, sizeof buf, f)) > 0) out->append(buf, n);
    const bool ok = !ferror(f);
    fclose(f);
    return ok;
}
// io::FileFingerprint (io.rs:23-45)
struct Fingerprint {
    std::string path;
    unsigned long long size = 0, modified = 0;
    bool operator==(const Fingerprint& o) const { return path == o.path && size == o.size && modified == o.modified; }
};
bool fingerprint(const std::string& path, Fingerprint* fp) {
    struct stat st;
    if (stat(path.c_str(), &st) != 0) return false;
    fp->path = absolute(path);
    fp->size = (unsigned long long)st.st_size;
    fp->modified = (unsigned long long)st.st_mtime;
    return true;
}

// io::Checkpoint (io.rs:47-90): raxtax.json, written like serde_json::to_writer_pretty
struct Checkpoint {
    std::string checkpoint_file, progress_file;
    Fingerprint db;
    bool raw_confidence = false, skip_exact_matches = false, tsv = false;
    bool both_strands = false;  // "strand": "both", written only in that mode (a plain run keeps the reference's key set)
    unsigned best_hits = 0;     // "best_hits": N, written only with --best-hits
    std::set<std::string> processed;  // #[serde(skip)]
};
std::string json_escape(const std::string& s) {
    std::string o;
    for (unsigned char c : s) {
        switch (c) {
            case '"': o += "\\\""; break;
            case '\\': o += "\\\\"; break;
            case '\n': o += "\\n"; break;
            case '\r': o += "\\r"; break;
            case '\t': o += "\\t"; break;
            default:
                if (c < 0x20) {
                    char b[8];
                    snprintf(b, sizeof b, "\\u%04x", c);
                    o += b;
                } else o += (char)c;
        }
    }
    return o;
}
bool checkpoint_save(const Checkpoint& c) {  // Checkpoint::save (io.rs:72-78): write raxtax.json.tmp, then rename
    const std::string tmp = std::filesystem::path(c.checkpoint_file).replace_extension("json.tmp").string();
    FILE* f = fopen(tmp.c_str(), "w");
    if (!f) return false;
    fprintf(f,
            "{\n  \"checkpoint_file\": \"%s\",\n  \"progress_file\": \"%s\",\n  \"db_fingerprint\": {\n    \"path\": \"%s\",\n"
            "    \"size\": %llu,\n    \"modified\": %llu\n  },\n  \"raw_confidence\": %s,\n  \"skip_exact_matches\": %s,\n  \"tsv\": %s%s%s\n}",
            json_escape(c.checkpoint_file).c_str(), json_escape(c.progress_file).c_str(), json_escape(c.db.path).c_str(), c.db.size,
            c.db.modified, c.raw_confidence ? "true" : "false", c.skip_exact_matches ? "true" : "false", c.tsv ? "true" : "false",
            c.both_strands ? ",\n  \"strand\": \"both\"" : "",
            c.best_hits ? (",\n  \"best_hits\": " + std::to_string(c.best_hits)).c_str() : "");
    if (fclose(f) != 0) return false;
    return rename(tmp.c_str(), c.checkpoint_file.c_str()) == 0;
}
// the handful of JSON this file needs: "key": "string" | number | true | false, nesting ignored (keys are unique across levels)
bool json_find(const std::string& j, const char* key, std::string* raw) {
    const std::string pat = std::string("\"") + key + "\"";
    size_t p = j.find(pat);
    if (p == std::string::npos) return false;
    p = j.find(':', p + pat.size());
    if (p == std::string::npos) return false;
    ++p;
    while (p < j.size() && isspace((unsigned char)j[p])) ++p;
    if (p >= j.size()) return false;
    if (j[p] == '"') {
        std::string o;
        for (++p; p < j.size() && j[p] != '"'; ++p) {
            if (j[p] == '\\' && p + 1 < j.size()) {
                ++p;
                switch (j[p]) {
                    case 'n': o += '\n'; break;
                    case 'r': o += '\r'; break;
                    case 't': o += '\t'; break;
                    case 'u':
                        if (p + 4 < j.size()) {  // \uXXXX, a surrogate pair for code points beyond the BMP -> UTF-8
                            unsigned long cp = strtoul(j.substr(p + 1, 4).c_str(), nullptr, 16);
                            p += 4;
                            if (cp >= 0xD800 && cp < 0xDC00 && p + 6 < j.size() && j[p + 1] == '\\' && j[p + 2] == 'u') {
                                const unsigned long lo = strtoul(j.substr(p + 3, 4).c_str(), nullptr, 16);
                                if (lo >= 0xDC00 && lo < 0xE000) {
                                    cp = 0x10000 + ((cp - 0xD800) << 10) + (lo - 0xDC00);
                                    p += 6;
                                }
                            }
                            if (cp < 0x80) o += (char)cp;
                            else if (cp < 0x800) {
                                o += (char)(0xC0 | (cp >> 6));
                                o += (char)(0x80 | (cp & 0x3F));
                            } else if (cp < 0x10000) {
                                o += (char)(0xE0 | (cp >> 12));
                                o += (char)(0x80 | ((cp >> 6) & 0x3F));
                                o += (char)(0x80 | (cp & 0x3F));
                            } else {
                                o += (char)(0xF0 | (cp >> 18));
                                o += (char)(0x80 | ((cp >> 12) & 0x3F));
                                o += (char)(0x80 | ((cp >> 6) & 0x3F));
                                o += (char)(0x80 | (cp & 0x3F));
                            }
                        }
                        break;
                    default: o += j[p];
                }
            } else o += j[p];
        }
        if (p >= j.size()) return false;
        *raw = o;
        return true;
    }
    size_t e = p;
    while (e < j.size() && j[e] != ',' && j[e] != '}' && !isspace((unsigned char)j[e])) ++e;
    *raw = j.substr(p, e - p);
    return !raw->empty();
}
bool checkpoint_load(const std::string& path, Checkpoint* c) {  // serde_json::from_reader (io.rs:208-209)
    std::string j, v;
    if (!read_raw(path, &j)) return false;
    auto b = [&](const char* k, bool* out) {
        if (!json_find(j, k, &v) || (v != "true" && v != "false")) return false;
        *out = v == "true";
        return true;
    };
    if (!json_find(j, "checkpoint_file", &c->checkpoint_file) || !json_find(j, "progress_file", &c->progress_file) ||
        !json_find(j, "path", &c->db.path))
        return false;
    if (!json_find(j, "size", &v)) return false;
    c->db.size = strtoull(v.c_str(), nullptr, 10);
    if (!json_find(j, "modified", &v)) return false;
    c->db.modified = strtoull(v.c_str(), nullptr, 10);
    c->both_strands = json_find(j, "strand", &v) && v == "both";
    c->best_hits = json_find(j, "best_hits", &v) ? (unsigned)strtoul(v.c_str(), nullptr, 10) : 0u;
    return b("raw_confidence", &c->raw_confidence) && b("skip_exact_matches", &c->skip_exact_matches) && b("tsv", &c->tsv);
}
// io::check_incomplete_output (io.rs:156-188): drop the result lines of queries the progress file does not list
bool check_incomplete_output(const std::string& path, const std::set<std::string>& processed) {
    std::ifstream in(path);
    if (!in) return false;
    std::vector<std::string> kept;
    bool needs_rewrite = false;
    std::string line;
    while (std::getline(in, line)) {
        const size_t tab = line.find('\t');
        if (tab != std::string::npos && processed.count(line.substr(0, tab))) kept.push_back(line);
        else if (tab != std::string::npos) needs_rewrite = true;
    }
    in.close();
    if (needs_rewrite) {
        const std::string tmp = std::filesystem::path(path).replace_extension("tmp").string();
        std::ofstream out(tmp, std::ios::trunc);
        for (size_t i = 0; i < kept.size(); ++i) out << (i ? "\n" : "") << kept[i];
        out << "\n";  // writeln!(tmp_file, "{}", retained_lines.join("\n"))
        out.close();
        if (!out || rename(tmp.c_str(), path.c_str()) != 0) return false;
    }
    return true;
}

}  // namespace

int main(int argc, char** argv) {
    Args a;
    for (int i = 1; i < argc; ++i) {
        std::string s = argv[i];
        auto val = [&](const char* name) -> const char* {
            if (i + 1 >= argc) {
                fprintf(stderr, "error: a value is required for '%s'\n", name);
                exit(EX_USAGE_);
            }
            return argv[++i];
        };
        if (s == "-d" || s == "--database-path") a.database_path = val("--database-path");
        else if (s == "-i" || s == "--query-file") a.query_file = val("--query-file");
        else if (s == "--skip-exact-matches") a.skip_exact_matches = true;
        else if (s == "--tsv") a.tsv = true;
        else if (s == "--only-db") a.only_db = true;
        else if (s == "--skip-db") a.skip_db = true;
        else if (s == "-c" || s == "--clean") a.clean = true;
        else if (s == "--raw-confidence") a.raw_confidence = true;
        else if (s == "-t" || s == "--threads") a.threads = atoi(val("--threads"));
        else if (s == "-o" || s == "--prefix") a.prefix = val("--prefix");
        else if (s == "--redo") a.redo = true;
        else if (s == "--pin") a.pin = true;
        else if (s == "--gpu") a.gpu = atoi(val("--gpu"));
        else if (s == "--gpus") a.gpus = std::max(1, atoi(val("--gpus")));
        else if (s == "--shard-references") a.shard_refs = true;
        else if (s == "--batch") a.batch = (size_t)atoll(val("--batch"));
        else if (s == "--strand") {  // vsearch's spelling
            const std::string v = val("--strand");
            if (v != "plus" && v != "both") {
                fprintf(stderr, "error: invalid value '%s' for '--strand <STRAND>'\n  [possible values: plus, both]\n", v.c_str());
                return EX_USAGE_;
            }
            a.both_strands = v == "both";
        }
        else if (s == "--best-hits") {
            const std::string v = val("--best-hits");
            const bool digits = !v.empty() && v.size() <= 2 && v.find_first_not_of("0123456789") == std::string::npos;
            const unsigned n = digits ? (unsigned)atoi(v.c_str()) : 0u;
            if (n < 1 || n > 64) {
                fprintf(stderr, "error: invalid value '%s' for '--best-hits <N>': a number in 1..64 is required\n", v.c_str());
                return EX_USAGE_;
            }
            a.best_hits = n;
        }
        else if (s == "--verbose") a.verbosity = std::min(5, a.verbosity + 1);  // clap_verbosity_flag::Verbosity<InfoLevel> (io.rs:152-153)
        else if (s == "--quiet") a.verbosity = std::max(0, a.verbosity - 1);
        else if (s.size() >= 2 && s[0] == '-' && s.find_first_not_of('v', 1) == std::string::npos) a.verbosity = std::min(5, a.verbosity + (int)s.size() - 1);  // -v, -vv, ...
        else if (s.size() >= 2 && s[0] == '-' && s.find_first_not_of('q', 1) == std::string::npos) a.verbosity = std::max(0, a.verbosity - ((int)s.size() - 1));
        else if (s == "-h" || s == "--help") {
            usage();
            return 0;
        } else {
            fprintf(stderr, "error: unexpected argument '%s'\n", s.c_str());
            usage();
            return EX_USAGE_;
        }
    }
    if (a.database_path.empty() || (a.query_file.empty() && !a.only_db)) {
        usage();
        return EX_USAGE_;
    }
    if (a.only_db && a.skip_db) {
        fprintf(stderr, "error: the argument '--only-db' cannot be used with '--skip-db'\n");
        return EX_USAGE_;
    }
    if (a.both_strands && a.shard_refs) {
        fprintf(stderr, "error: the argument '--strand both' cannot be used with '--shard-references'\n");
        return EX_USAGE_;
    }
    if (a.best_hits && a.shard_refs) {
        fprintf(stderr, "error: the argument '--best-hits' cannot be used with '--shard-references'\n");
        return EX_USAGE_;
    }
    // ---- Args::get_output (io.rs:202-263): checkpoint, output folder, writers ----------------------------------------
    const std::string ckp_path = a.prefix + "/raxtax.json", out_path = a.prefix + "/raxtax.out", tsv_path = a.prefix + "/raxtax.tsv",
                      hits_path = a.prefix + "/raxtax.hits";
    Checkpoint ckp;
    auto checkpoint_new = [&](Checkpoint* c) {  // Checkpoint::new (io.rs:60-70)
        *c = Checkpoint();
        c->checkpoint_file = absolute(ckp_path);
        c->progress_file = std::filesystem::path(absolute(ckp_path)).replace_extension("ckp").string();
        c->raw_confidence = a.raw_confidence;
        c->skip_exact_matches = a.skip_exact_matches;
        c->tsv = a.tsv;
        c->both_strands = a.both_strands;
        c->best_hits = a.best_hits;
        return fingerprint(a.database_path, &c->db);
    };
    bool resumed = false;
    if (!a.redo && is_file(ckp_path)) {
        Checkpoint old;
        if (checkpoint_load(ckp_path, &old)) {
            Fingerprint now;
            const bool valid = fingerprint(old.db.path, &now) && a.tsv == old.tsv && a.raw_confidence == old.raw_confidence &&
                               a.skip_exact_matches == old.skip_exact_matches && a.both_strands == old.both_strands && a.best_hits == old.best_hits &&
                               now == old.db;  // checkpoint_valid (io.rs:288-303)
            if (valid) {
                std::ifstream prog(old.progress_file);
                std::string line;
                while (std::getline(prog, line)) old.processed.insert(line);
                if (!check_incomplete_output(out_path, old.processed) || (a.tsv && !check_incomplete_output(tsv_path, old.processed)) ||
                    (a.best_hits && is_file(hits_path) && !check_incomplete_output(hits_path, old.processed))) {
                    fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m cannot repair the output files under %s\n", a.prefix.c_str());
                    return EX_CANTCREAT_;
                }
                ckp = old;
                resumed = true;
            }
        } else {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to read checkpoint!\n");
        }
    }
    if (!resumed && !checkpoint_new(&ckp)) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to parse %s: cannot read file\n", a.database_path.c_str());
        return EX_CANTCREAT_;
    }
    if (is_dir(a.prefix) && !is_file(ckp_path) && !a.redo) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Output folder %s already exists! Please specify another folder with -o <PATH> or run with --redo to force overriding existing files!\n",
                a.prefix.c_str());
        return EX_CANTCREAT_;
    }
    {
        std::error_code ec;
        std::filesystem::create_directories(a.prefix, ec);
        if (ec) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m cannot create %s\n", a.prefix.c_str());
            return EX_CANTCREAT_;
        }
    }
    const char* mode = a.redo ? "w" : "a";  // create_file(path, append = !redo) (io.rs:190-199)
    const bool restart_note = !a.redo && exists(ckp_path) && a.verbosity >= 3;
    Writers w;
    w.verbosity = a.verbosity;
    if (a.tsv) w.tsv = fopen(tsv_path.c_str(), mode);
    if (a.best_hits) w.hits = fopen(hits_path.c_str(), mode);
    w.log = fopen((a.prefix + "/raxtax.log").c_str(), mode);
    if (w.log && restart_note) {
        fprintf(w.log, "[INFO ] Restarting from checkpoint %s\n", ckp.checkpoint_file.c_str());
        fprintf(stderr, "[INFO ] Restarting from checkpoint %s\n", ckp.checkpoint_file.c_str());
    }
    w.primary = fopen(out_path.c_str(), mode);
    w.progress = fopen((a.prefix + "/raxtax.ckp").c_str(), mode);
    if (!w.primary || !w.log || !w.progress || (a.tsv && !w.tsv) || (a.best_hits && !w.hits)) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m cannot create output files under %s\n", a.prefix.c_str());
        return EX_CANTCREAT_;
    }
    {  // io::write_build_info (io.rs:92-110)
        std::string cmd;
        for (int i = 0; i < argc; ++i) cmd += std::string(i ? " " : "") + argv[i];
        fprintf(w.log, "raxtax-b200 1.5.0 (B200 sm_100a build of the raxtax hot path)\nBuild flags: \nCommand: %s\n"
                       "------------------------------------------------------------\n", cmd.c_str());
        fflush(w.log);
    }
    auto t_total = std::chrono::steady_clock::now();

    // ---- parser::parse_reference_fasta_file (parser.rs:37-44) on the checkpoint's database path (main.rs:61) ----------------
    rxh_tree* tree = nullptr;
    bool store_db = false;
    {
        if (a.verbosity >= 3) fprintf(stderr, "[INFO ] Trying to read from database file...\n");
        int was_database = 0;
        tree = rxh_tree_from_file(ckp.db.path.c_str(), &was_database);  // parser::parse_reference_fasta_file (parser.rs:37-44)
        if (!tree) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to parse %s: %s\n", ckp.db.path.c_str(), rxh_last_error());
            return EX_NOINPUT_;
        }
        store_db = !was_database;
    }
    std::string created_db;
    if (store_db && !a.skip_db) {  // main.rs:73-98, Args::get_db_output (io.rs:269-286)
        std::filesystem::path name = std::filesystem::path(a.database_path).filename();
        if (name.empty()) name = "database";
        const std::string db_path = (std::filesystem::path(a.prefix) / name).replace_extension("bin").string();
        if (is_file(db_path) && !a.redo) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Could not create database! Rerun with --skip-db to skip this step.: Output database file %s already exists! Delete it or run with --redo to force overriding existing files!\n",
                    db_path.c_str());
            return EX_CANTCREAT_;
        }
        if (a.verbosity >= 3) {
            fprintf(w.log, "[INFO ] Created binary database at %s\n", db_path.c_str());
            fprintf(stderr, "[INFO ] Writing database to file...\n");
        }
        if (rxh_tree_save_bin(tree, db_path.c_str()) != 0) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to write database: %s\n", rxh_last_error());
            return EX_IOERR_;
        }
        created_db = absolute(db_path);
        Fingerprint fp;
        if (!fingerprint(db_path, &fp) || (ckp.db = fp, !checkpoint_save(ckp)))
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to write checkpoint! Continuing without...\n");
    } else if (!checkpoint_save(ckp)) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to write checkpoint! Continuing without...\n");
    }
    if (a.only_db) return EX_OK_;

    // ---- parser::parse_query_fasta_file with the processed queries skipped (main.rs:104-117) ------------------------------
    rxh_queries* queries = rxh_queries_from_file(a.query_file.c_str());
    if (!queries) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Failed to parse %s: %s\n", a.query_file.c_str(), rxh_last_error());
        return EX_NOINPUT_;
    }
    if (!ckp.processed.empty()) {
        std::string blob;
        for (const auto& l : ckp.processed) blob += l + "\n";
        rxh_queries_skip(queries, blob.data(), blob.size());
    }

    // one context per GPU: the index replicated on each (BASELINE config 3: query-partitioned, no collective), or with
    // --shard-references a contiguous 1/N of the lineage-sorted references on each (config 5)
    const bool sharded = a.shard_refs && a.gpus > 1;
    std::vector<uint64_t> cuts;
    if (sharded) {
        const uint64_t n = rxh_tree_num_tips(tree);
        cuts.push_back(0);
        for (int r = 1; r < a.gpus; ++r) cuts.push_back(std::max<uint64_t>(n * (uint64_t)r / (uint64_t)a.gpus / 32 * 32, cuts.back() + 1));
        cuts.push_back(n);
        if (n < (uint64_t)a.gpus) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m --shard-references: fewer references than GPUs\n");
            return EX_USAGE_;
        }
    }
    std::vector<rtx_ctx*> ctxs((size_t)a.gpus, nullptr);
    for (int g = 0; g < a.gpus; ++g) {
        if (rtx_ctx_create(a.gpu + g, &ctxs[(size_t)g]) != 0) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m %s\n", rtx_last_error(nullptr));
            return EX_TEMPFAIL_;
        }
        if ((sharded ? rxh_tree_upload_sharded(tree, ctxs[(size_t)g], (uint32_t)a.gpus, (uint32_t)g, cuts.data())
                     : rxh_tree_upload(tree, ctxs[(size_t)g], 0, 0)) != 0) {
            fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m index upload: %s\n", rxh_last_error());
            return EX_TEMPFAIL_;
        }
    }
    int warnings = 0;
    auto t0 = std::chrono::steady_clock::now();
    int rc = sharded ? rxh_raxtax_sharded(ctxs.data(), ctxs.size(), queries, tree, a.skip_exact_matches, a.raw_confidence, a.batch, send_cb, &w,
                                          a.tsv, log_cb, &w, &warnings)
                     : a.best_hits ? rxh_raxtax_best_hits(ctxs.data(), ctxs.size(), queries, tree, a.skip_exact_matches, a.raw_confidence, a.batch,
                                                          send_cb, &w, a.tsv, log_cb, &w, &warnings, a.both_strands, a.best_hits, hits_cb, &w)
                     : (a.both_strands ? rxh_raxtax_both_strands : rxh_raxtax_multi)(ctxs.data(), ctxs.size(), queries, tree, a.skip_exact_matches,
                                                                                     a.raw_confidence, a.batch, send_cb, &w, a.tsv, log_cb, &w, &warnings);
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    if (!w.commit() && rc == 0) {  // the labels still held back: results first, then progress
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Could not write the result files\n");
        return EX_IOERR_;
    }
    if (rc != 0) {
        fprintf(stderr, "\x1b[31m[ERROR]\x1b[0m Error while sending results to IO-thread!: %s\n", rxh_last_error());
        return EX_TEMPFAIL_;
    }
    if (warnings && a.verbosity >= 2)
        fprintf(stderr, "\x1b[33m[WARN ]\x1b[0m Exact matches for some queries differ above the species level! Check the log file for more information!\n");
    if (a.verbosity >= 3) {
        fprintf(w.log, "[INFO ] raxtax(), Elapsed=%.6fs\n", secs);
        fprintf(w.log, "[INFO ] Total Runtime, Elapsed=%.6fs\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t_total).count());
    }
    for (FILE* f : {w.primary, w.tsv, w.log, w.progress, w.hits})
        if (f) fclose(f);
    if (a.clean) {  // Checkpoint::cleanup (io.rs:80-89); the database only if it lives under PREFIX as <stem>.bin (see the header)
        if (a.verbosity >= 3) fprintf(stderr, "[INFO ] Removing checkpoint files...\n");
        remove(ckp.checkpoint_file.c_str());
        remove(ckp.progress_file.c_str());
        const std::string pre = absolute(a.prefix) + "/";
        if (ckp.db.path.compare(0, pre.size(), pre) == 0 && ckp.db.path.size() > 4 && ckp.db.path.compare(ckp.db.path.size() - 4, 4, ".bin") == 0)
            remove(ckp.db.path.c_str());
    }
    rxh_queries_free(queries);
    rxh_tree_free(tree);
    for (rtx_ctx* c : ctxs) rtx_ctx_destroy(c);
    return EX_OK_;
}
