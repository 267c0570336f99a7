// zarc-b200: the reference CLI's pack / unpack / list-files (crates/zarc-cli/src/{pack,unpack,
// list_files}.rs) over the GPU content path.  File contents are gathered into pinned batches and go
// through zg_pack_batch / zg_unpack_batch; the walk, the metadata and the ordered writes stay here.
#include <algorithm>
#include <cerrno>
#include <cstring>
#include <fcntl.h>
#include <filesystem>
#include <memory>
#include <regex>
#include <string>
#include <sys/stat.h>
#include <sys/time.h>
#include <unistd.h>
#include <vector>

#include "zarc_host.hpp"
#include "zarcgpu_dl.hpp"

namespace fs = std::filesystem;
using namespace zarc;

// $ZARC_TIMING=1: wall-clock of the phases on stderr
static double now_s() {
	timespec ts;
	clock_gettime(CLOCK_MONOTONIC, &ts);
	return (double)ts.tv_sec + 1e-9 * (double)ts.tv_nsec;
}
// page-locking a buffer costs about as much as copying it a few times: only worth it for multi-pass jobs
static const uint64_t PIN_THRESHOLD = 1ull << 30;
static const bool TIMING = getenv("ZARC_TIMING") != nullptr;
static double t_last = now_s();
static void lap(const char* what) {
	if (!TIMING) return;
	double t = now_s();
	fprintf(stderr, "[timing] %-28s %8.1f ms\n", what, (t - t_last) * 1e3);
	t_last = t;
}

// content bytes gathered before one GPU pass ($ZARC_BATCH_MB overrides; tests use it to force several passes)
static const uint64_t BATCH_BYTES = getenv("ZARC_BATCH_MB") ? (uint64_t)atoll(getenv("ZARC_BATCH_MB")) << 20 : 1ull << 30;

[[noreturn]] static void usage(int code) {
	fprintf(code ? stderr : stdout,
	        "zarc-b200 -- zarc archives with the content path on the GPU\n\n"
	        "  zarc-b200 pack --output <PATH> [--level <N>] [--zstd <name=value>]... [-L|--follow-symlinks] <PATHS>...\n"
	        "  zarc-b200 unpack [--filter <REGEX>]... [--verify <DIGEST>] <PATH>\n"
	        "  zarc-b200 list-files [--only-files] [--decorate] [--filter <REGEX>]... <PATH>\n\n"
	        "  --level: -131072 to 22 (default 3).  Negative levels store literals uncompressed and sample the input:\n"
	        "           larger archives; -1 packs faster than 1, -2 to -4 are no faster than -1, -5 and below faster again\n");
	exit(code);
}

// --zstd name=value: the names zarc-cli accepts (pack.rs:140-195)
static bool parse_zstd_param(const std::string& kv, ZstdParameter& p, int& v) {
	size_t eq = kv.find('=');
	std::string name = kv.substr(0, eq), val = eq == std::string::npos ? "1" : kv.substr(eq + 1);
	std::string low;
	for (char c : name) low += (char)tolower((unsigned char)c);
	static const struct { const char* n; ZstdParameter p; } names[] = {
	    {"compressionlevel", ZstdParameter::CompressionLevel}, {"windowlog", ZstdParameter::WindowLog}, {"hashlog", ZstdParameter::HashLog},
	    {"chainlog", ZstdParameter::ChainLog}, {"searchlog", ZstdParameter::SearchLog}, {"minmatch", ZstdParameter::MinMatch},
	    {"targetlength", ZstdParameter::TargetLength}, {"strategy", ZstdParameter::Strategy}, {"contentsizeflag", ZstdParameter::ContentSizeFlag},
	    {"checksumflag", ZstdParameter::ChecksumFlag}, {"dictidflag", ZstdParameter::DictIdFlag}};
	for (auto& e : names)
		if (low == e.n) {
			p = e.p;
			if (val == "true") v = 1;
			else if (val == "false") v = 0;
			else v = atoi(val.c_str());
			return true;
		}
	return false;
}

// ------------------------------------------------------------------------------------------------
struct PendingEntry {
	File file;
	bool has_content = false;
	size_t content_index = 0;
};

static int cmd_pack(int argc, char** argv) {
	std::string output;
	std::vector<std::string> paths;
	std::vector<std::pair<ZstdParameter, int>> params;
	int level = 0;
	bool have_level = false, follow = false;
	for (int i = 0; i < argc; i++) {
		std::string a = argv[i];
		auto need = [&](const char* what) -> std::string {
			if (i + 1 >= argc) {
				fprintf(stderr, "error: %s needs a value\n", what);
				usage(2);
			}
			return argv[++i];
		};
		if (a == "--output" || a == "-o") output = need("--output");
		else if (a == "--level") { level = atoi(need("--level").c_str()); have_level = true; }
		else if (a == "--zstd") {
			ZstdParameter p; int v;
			std::string kv = need("--zstd");
			if (!parse_zstd_param(kv, p, v)) { fprintf(stderr, "error: unknown zstd parameter %s\n", kv.c_str()); return 2; }
			params.emplace_back(p, v);
		} else if (a == "-L" || a == "--follow-symlinks") follow = true;
		else if (a == "--store") { fprintf(stderr, "error: --store is not supported (the reference's uncompressed frames are not valid Zstandard)\n"); return 2; }
		else if (!a.empty() && a[0] == '-') { fprintf(stderr, "error: unknown option %s\n", a.c_str()); usage(2); }
		else paths.push_back(a);
	}
	if (output.empty() || paths.empty()) usage(2);
	std::FILE* out = fopen(output.c_str(), "wb");
	if (!out) { fprintf(stderr, "error: %s: %s\n", output.c_str(), strerror(errno)); return 1; }
	lap("start");
	Encoder zarc(out);
	lap("encoder (context) create");
	zarc.set_zstd_parameter(ZstdParameter::ChecksumFlag, 1);  // pack.rs:227-228
	if (have_level) zarc.set_zstd_parameter(ZstdParameter::CompressionLevel, level);
	for (auto& pv : params) zarc.set_zstd_parameter(pv.first, pv.second);

	GpuLib& g = gpu();
	// the walk (WalkDir order: a root first, then its contents in directory order, pack.rs:246)
	struct Walked {
		std::string path;
		bool regular;
		uint64_t size;
	};
	std::vector<Walked> walked;
	uint64_t total_content = 0;
	auto note = [&](const std::string& path, const fs::file_status& st) {
		bool reg = fs::is_regular_file(st);
		uint64_t sz = 0;
		if (reg) {
			std::error_code ec2;
			sz = (uint64_t)fs::file_size(path, ec2);
			if (ec2) sz = 0;
		}
		walked.push_back({path, reg, sz});
		total_content += sz;
	};
	for (const std::string& root : paths) {
		std::error_code ec;
		fs::file_status rs = follow ? fs::status(root, ec) : fs::symlink_status(root, ec);
		if (ec) { fprintf(stderr, "read error: %s: %s\n", root.c_str(), ec.message().c_str()); continue; }
		note(root, rs);
		if (!fs::is_directory(rs)) continue;
		auto opts = follow ? fs::directory_options::follow_directory_symlink : fs::directory_options::none;
		for (auto it = fs::recursive_directory_iterator(root, opts | fs::directory_options::skip_permission_denied, ec);
		     it != fs::recursive_directory_iterator(); it.increment(ec)) {
			if (ec) { fprintf(stderr, "read error: %s\n", ec.message().c_str()); break; }
			fs::file_status st = follow ? it->status(ec) : it->symlink_status(ec);
			if (ec) { fprintf(stderr, "read error: %s: %s\n", it->path().c_str(), ec.message().c_str()); continue; }
			note(it->path().string(), st);
		}
	}
	lap("walk");
	// the batch buffer: page-locked when the job is large enough for the locking to pay for itself
	uint64_t batch_cap = std::min<uint64_t>(BATCH_BYTES, total_content + (1 << 16));
	bool pinned = total_content > PIN_THRESHOLD;
	std::unique_ptr<uint8_t[]> pageable;
	uint8_t* blob = nullptr;
	if (pinned) blob = (uint8_t*)g.zg_alloc_pinned(batch_cap + 1);
	else {
		pageable.reset(new uint8_t[batch_cap + 1]);  // not zero-filled
		blob = pageable.get();
	}
	if (!blob) { fprintf(stderr, "error: cannot allocate the batch buffer\n"); return 1; }
	lap("batch buffer");
	std::vector<uint8_t> big;  // a single file larger than a batch goes on its own
	std::vector<uint64_t> offs, lens;
	std::vector<PendingEntry> pending;
	uint64_t used = 0;
	auto flush = [&]() {
		lap("walk + read files");
		std::vector<Digest> digests = zarc.add_data_frames(blob, offs.data(), lens.data(), offs.size());
		lap("add_data_frames (GPU + write)");
		for (auto& pe : pending) {
			if (pe.has_content) pe.file.digest = digests[pe.content_index];
			zarc.add_file_entry(std::move(pe.file));
		}
		pending.clear();
		offs.clear();
		lens.clear();
		used = 0;
	};
	auto visit = [&](const std::string& filename, bool is_regular) {
		PendingEntry pe;
		pe.file = zarc.build_file_with_metadata(filename, follow);
		if (is_regular) {
			int fd = open(filename.c_str(), O_RDONLY);
			if (fd < 0) throw Error(filename + ": " + strerror(errno));
			struct stat st;
			fstat(fd, &st);
			uint64_t n = (uint64_t)st.st_size;
			if (n > batch_cap) {  // oversized: flush what is pending, then this file alone from pageable memory
				flush();
				big.resize(n);
				uint64_t done = 0;
				while (done < n) {
					ssize_t k = read(fd, big.data() + done, n - done);
					if (k <= 0) break;
					done += (uint64_t)k;
				}
				close(fd);
				pe.file.digest = zarc.add_data_frame(big.data(), done);
				big.clear();
				big.shrink_to_fit();
				zarc.add_file_entry(std::move(pe.file));
				return;
			}
			if (used + n > batch_cap) flush();
			uint64_t done = 0;
			while (done < n) {
				ssize_t k = read(fd, blob + used + done, n - done);
				if (k <= 0) break;
				done += (uint64_t)k;
			}
			close(fd);
			pe.has_content = true;
			pe.content_index = offs.size();
			offs.push_back(used);
			lens.push_back(done);
			used += done;
		}
		pending.push_back(std::move(pe));
	};
	try {
		for (const Walked& w : walked) visit(w.path, w.regular);
		flush();
		Digest digest = zarc.finalise();
		lap("finalise");
		if (pinned) g.zg_free_pinned(blob);
		fclose(out);
		printf("digest: %s\n", digest.base64().c_str());
	} catch (const std::exception& e) {
		if (pinned) g.zg_free_pinned(blob);
		fclose(out);
		fprintf(stderr, "error: %s\n", e.what());
		return 1;
	}
	return 0;
}

// ------------------------------------------------------------------------------------------------
static bool matches(const std::vector<std::regex>& filters, const std::string& name) {
	if (filters.empty()) return true;
	for (auto& f : filters)
		if (std::regex_search(name, f)) return true;
	return false;
}

// metadata/decode.rs: ownership (best effort), permissions, timestamps
static void set_metadata(const File& entry, const std::string& path) {
	if (entry.user || entry.group) {
		uid_t uid = entry.user && entry.user->id ? (uid_t)*entry.user->id : (uid_t)-1;
		gid_t gid = entry.group && entry.group->id ? (gid_t)*entry.group->id : (gid_t)-1;
		if (chown(path.c_str(), uid, gid) != 0 && errno != EPERM) fprintf(stderr, "warning: chown %s: %s\n", path.c_str(), strerror(errno));
	}
	// setuid / setgid bits of an untrusted archive are not restored (the reference applies the mode verbatim)
	if (entry.mode && chmod(path.c_str(), *entry.mode & 01777) != 0) fprintf(stderr, "warning: chmod %s: %s\n", path.c_str(), strerror(errno));
	if (entry.timestamps) {
		timespec ts[2];
		ts[0].tv_nsec = ts[1].tv_nsec = UTIME_OMIT;
		ts[0].tv_sec = ts[1].tv_sec = 0;
		if (entry.timestamps->accessed) ts[0] = timespec{(time_t)entry.timestamps->accessed->secs, (long)entry.timestamps->accessed->nanos};
		if (entry.timestamps->modified) ts[1] = timespec{(time_t)entry.timestamps->modified->secs, (long)entry.timestamps->modified->nanos};
		if (utimensat(AT_FDCWD, path.c_str(), ts, 0) != 0) fprintf(stderr, "warning: utimens %s: %s\n", path.c_str(), strerror(errno));
	}
}

static int cmd_unpack(int argc, char** argv) {
	std::string input, verify;
	std::vector<std::regex> filters;
	for (int i = 0; i < argc; i++) {
		std::string a = argv[i];
		if (a == "--filter" && i + 1 < argc) filters.emplace_back(argv[++i]);
		else if (a == "--verify" && i + 1 < argc) verify = argv[++i];
		else if (!a.empty() && a[0] == '-') { fprintf(stderr, "error: unknown option %s\n", a.c_str()); usage(2); }
		else input = a;
	}
	if (input.empty()) usage(2);
	try {
		lap("start");
		Decoder zarc = Decoder::open(input);
		lap("decoder (context) create");
		if (!verify.empty()) {
			if (Digest::from_base64(verify) != zarc.trailer().digest) {
				fprintf(stderr, "integrity failure: zarc file digest is %s\n", zarc.trailer().digest.base64().c_str());
				return 1;
			}
		} else fprintf(stderr, "digest: %s\n", zarc.trailer().digest.base64().c_str());
		zarc.read_directory();
		uint64_t unpacked = 0, skipped = 0;
		std::vector<const File*> batch;
		std::vector<Digest> digests;
		uint64_t batch_bytes = 0;
		auto flush = [&]() {
			if (batch.empty()) return;
			std::vector<ContentFrame> frames = zarc.read_content_frames(digests);
			for (size_t i = 0; i < batch.size(); i++) {
				std::string path = *batch[i]->name.to_safe_path();  // checked when the entry was queued
				fs::path parent = fs::path(path).parent_path();
				if (!parent.empty()) fs::create_directories(parent);  // in case its entry wasn't in the zarc
				std::FILE* f = fopen(path.c_str(), "wb");
				if (!f) throw Error(path + ": " + strerror(errno));
				if (!frames[i].data.empty() && fwrite(frames[i].data.data(), 1, frames[i].data.size(), f) != frames[i].data.size()) {
					fclose(f);
					throw Error(path + ": write failed");
				}
				fclose(f);
				if (!frames[i].verified.value_or(false)) fprintf(stderr, "error: frame verification failed! path=%s\n", path.c_str());  // only logged: unpack.rs:118-120
				set_metadata(*batch[i], path);
				unpacked++;
			}
			batch.clear();
			digests.clear();
			batch_bytes = 0;
		};
		for (const File& entry : zarc.files()) {
			std::string shown = entry.name.to_path();
			if (!matches(filters, shown)) continue;
			std::optional<std::string> safe = entry.name.to_safe_path();
			if (!safe) {
				// never write outside the extraction directory: "..", absolute and '/'-holding components are refused
				fprintf(stderr, "warning: skipping entry with unsafe path: %s\n", shown.c_str());
				skipped++;
				continue;
			}
			const std::string& name = *safe;
			if (entry.is_dir()) {
				fs::create_directories(name);
				set_metadata(entry, name);
			} else if (entry.is_normal()) {
				const Frame* fr = zarc.frame(*entry.digest);
				if (!fr) {
					fprintf(stderr, "warning: frame not found\n");
					continue;
				}
				if (batch_bytes + fr->uncompressed > BATCH_BYTES) flush();
				batch.push_back(&entry);
				digests.push_back(*entry.digest);
				batch_bytes += fr->uncompressed;
			}
		}
		flush();
		lap("read_content_frames (GPU) + write files");
		fprintf(stderr, "unpacked %llu files\n", (unsigned long long)unpacked);
		if (skipped) fprintf(stderr, "skipped %llu entries with unsafe paths\n", (unsigned long long)skipped);
	} catch (const std::exception& e) {
		fprintf(stderr, "error: %s\n", e.what());
		return 1;
	}
	return 0;
}

static int cmd_list_files(int argc, char** argv) {
	std::string input;
	std::vector<std::regex> filters;
	bool only_files = false;
	for (int i = 0; i < argc; i++) {
		std::string a = argv[i];
		if (a == "--filter" && i + 1 < argc) filters.emplace_back(argv[++i]);
		else if (a == "--only-files") only_files = true;
		else if (a == "--decorate") {}  // parsed and ignored, suffixes are always printed: list_files.rs:24-25,51-57
		else if (!a.empty() && a[0] == '-') { fprintf(stderr, "error: unknown option %s\n", a.c_str()); usage(2); }
		else input = a;
	}
	if (input.empty()) usage(2);
	try {
		Decoder zarc = Decoder::open(input);
		zarc.read_directory();
		for (const File& entry : zarc.files()) {
			if (only_files && entry.special) continue;
			std::string name = entry.name.to_path();
			if (!matches(filters, name)) continue;
			const char* suffix = entry.is_dir() ? "/" : entry.is_symlink() ? "@" : entry.is_hardlink() ? "#" : "";
			printf("%s%s\n", name.c_str(), suffix);
		}
	} catch (const std::exception& e) {
		fprintf(stderr, "error: %s\n", e.what());
		return 1;
	}
	return 0;
}

int main(int argc, char** argv) {
	if (argc < 2) usage(2);
	std::string cmd = argv[1];
	if (cmd == "-h" || cmd == "--help" || cmd == "help") usage(0);
	try {
		if (cmd == "pack") return cmd_pack(argc - 2, argv + 2);
		if (cmd == "unpack") return cmd_unpack(argc - 2, argv + 2);
		if (cmd == "list-files") return cmd_list_files(argc - 2, argv + 2);
	} catch (const std::exception& e) {
		fprintf(stderr, "error: %s\n", e.what());
		return 1;
	}
	fprintf(stderr, "error: unknown command %s\n", cmd.c_str());
	usage(2);
}
