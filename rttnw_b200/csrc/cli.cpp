// cli.cpp — `rttnw <scene>`: the reference's CLI (src/main.rs:236-258) on top of the C ABI.
// Same positional argument, same usage text, same stdout lines, writes image.png (RGBA8) in the
// CWD and reads assets/earth.png relative to it. Optional flags default to the reference values:
//   --spp N  --width W  --height H  --seed S  --scene-seed S  --gpus N  --out PATH  --chunk N
//   --checkpoint PATH [--checkpoint-every K]  --resume PATH  --stop-after-chunks N
//   --adaptive THRESHOLD [--min-spp N] [--step N]
// --adaptive (one GPU; rtx_render_adaptive): every 8x4 tile stops sampling once its noise estimate is below THRESHOLD,
// with --spp as the most samples a pixel gets; --min-spp defaults to spp / 64 (at least 2, even), --step to --min-spp.
// It prints the samples spent and the tiles that converged. Not with --gpus > 1, --checkpoint or --resume: several GPUs
// would have to decide on their combined buffer every round.
// Checkpoint / resume (the reference keeps pixels in RAM until the final save_buffer, main.rs:202-231, so a
// killed 10k-spp render loses everything): after every K chunks each GPU writes its fp32 accumulator and the
// next sample index it would render to PATH.<gpu>; --resume reloads them (same scene, size, spp, seed, gpus)
// and carries on. Samples are keyed by their global index, so a resumed image equals an uninterrupted one up
// to fp32 summation order.
// --gpus N. What costs time on a multi-GPU box is not the render but bringing CUDA up (measured on an 8 x B200 box,
// profiles/r2_cli_wallclock.txt): 0.8 s per VISIBLE device in one process (6.6 s with all eight, whether one context
// is created or eight), and processes that initialise at the same time queue behind each other (8 processes, each seeing
// one device: the last one is up after 9.4 s) — against 1.3 s for the 10 000-spp final scene on eight GPUs. So:
//   * every process sees ONLY its device (CUDA_VISIBLE_DEVICES is narrowed before its first CUDA call): one GPU is up
//     in 0.9 s instead of 6.6 s;
//   * the parent brings its own device up first, alone, THEN starts one worker process per further device (fork + exec
//     of this binary with --worker) and begins to render at once; the workers bring CUDA up one after the other behind
//     it, each waiting for the previous one (start-ups that overlap all finish together, after ~1.1 s x their number);
//   * the samples are not divided in advance: every process claims chunks of global sample indices from a counter in
//     a shared mapping until none are left, so a device that is up early renders more, and a device that is not up by
//     the time the frame is finished is not waited for (the parent ends it). Samples are keyed by their global index, so
//     the frame is the same whichever process rendered what (up to fp32 summation order);
//   * processes that see one device each cannot map each other's memory, so the end-of-frame combine goes through the
//     host: a worker copies its accumulator (10 MB at 800x800) into the shared mapping, the parent uploads the
//     accumulators that hold samples and runs the fused sum + tonemap kernel on local copies (milliseconds per frame).
// With --checkpoint / --resume (which need the sample ranges of a rank to be contiguous), or RTTNW_SINGLE_PROCESS=1,
// one process drives the N devices with a thread each, static ranges and the peer-mapped combine over NVLink.
#include <signal.h>
#include <sys/mman.h>
#include <sys/wait.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstdint>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#include "rttnw_b200.h"

static void usage(const char* argv0) {  // main.rs:239-249
    std::fprintf(stderr, "Usage: %s <scene>\n", argv0);
    std::fprintf(stderr, "Possible scenes:\n");
    static const char* names[] = {"random_scene", "two_spheres", "two_perlin_spheres", "earth", "simple_light",
                                  "empty_cornell_box", "cornell_box", "smoke_cornell_box", "final_scene"};
    for (int i = 0; i < 9; ++i) std::fprintf(stderr, "\t- %d: %s\n", i + 1, names[i]);
}

#define RTX(call)                                                            \
    do {                                                                     \
        if ((call) != RTX_OK) {                                              \
            std::fprintf(stderr, "%s failed: %s\n", #call, rtx_last_error()); \
            return 1;                                                        \
        }                                                                    \
    } while (0)

struct Rank {
    rtx_ctx* ctx = nullptr;
    rtx_scene* scene = nullptr;
    float* accum = nullptr;
    int rc = 0;
};

struct CheckpointHeader {  // little-endian, followed by width * height float4
    char magic[8];         // "RTXACC1"
    int32_t scene, width, height, spp_total, gpus, rank, next_sample, max_depth;
    uint64_t seed, scene_seed;
};

static bool write_checkpoint(const std::string& path, const CheckpointHeader& h, const std::vector<float>& acc) {
    std::string tmp = path + ".tmp";
    FILE* f = std::fopen(tmp.c_str(), "wb");
    if (!f) return false;
    bool ok = std::fwrite(&h, sizeof(h), 1, f) == 1 && std::fwrite(acc.data(), sizeof(float), acc.size(), f) == acc.size();
    ok = std::fclose(f) == 0 && ok;
    return ok && std::rename(tmp.c_str(), path.c_str()) == 0;  // never leaves a torn file behind
}
static bool read_checkpoint(const std::string& path, CheckpointHeader& h, std::vector<float>& acc) {
    FILE* f = std::fopen(path.c_str(), "rb");
    if (!f) return false;
    bool ok = std::fread(&h, sizeof(h), 1, f) == 1 && std::memcmp(h.magic, "RTXACC1", 8) == 0 && h.width > 0 && h.height > 0;
    if (ok) {
        acc.resize((size_t)h.width * h.height * 4);
        ok = std::fread(acc.data(), sizeof(float), acc.size(), f) == acc.size();
    }
    std::fclose(f);
    return ok;
}

// Narrows CUDA_VISIBLE_DEVICES to the `rank`-th device the user could see (`list`: the user's own CUDA_VISIBLE_DEVICES,
// empty = all devices). Must run before the first CUDA call of the process; the device is then number 0.
static void see_only_device(const std::string& list, int rank) {
    std::string pick = std::to_string(rank);
    if (!list.empty()) {
        size_t pos = 0;
        for (int i = 0; i < rank && pos != std::string::npos; ++i) {
            pos = list.find(',', pos);
            if (pos != std::string::npos) ++pos;
        }
        if (pos == std::string::npos || pos >= list.size()) pick = "no-such-device";  // fewer entries than ranks: rtx_ctx_create will say so
        else {
            size_t end = list.find(',', pos);
            pick = list.substr(pos, end == std::string::npos ? std::string::npos : end - pos);
        }
    }
    setenv("CUDA_VISIBLE_DEVICES", pick.c_str(), 1);
}

// What the processes of one multi-GPU render share (an anonymous memory file, inherited across exec).
struct SharedFrame {
    std::atomic<int> next_sample;  // first global sample index nobody has claimed yet
    std::atomic<int> state[16];    // per rank: 0 not up yet, 1 claiming / rendering, 2 finished (accumulator in its slot, if it has samples)
    std::atomic<int> samples[16];  // per rank: samples per pixel it rendered
    int rc[16];
    char pad[64];
    // followed by (gpus - 1) accumulators of width * height float4, rank r in slot r - 1
};

int main(int argc, char** argv) {
    int scene = -1, spp = -1, width = -1, height = -1, gpus = 1, chunk = 256, ckpt_every = 1, stop_after = -1;
    std::string ckpt_path, resume_path;
    unsigned long long seed = 1, scene_seed = 0;
    bool have_scene_seed = false;
    std::string out = "image.png";
    double adaptive = -1.0;  // --adaptive THRESHOLD (< 0: uniform sampling)
    int min_spp = -1, step_spp = -1;
    int worker_rank = -1, shm_fd = -1;  // --worker R --shm-fd FD --device-list L: a worker process of a multi-GPU render (internal)
    std::string device_list = std::getenv("CUDA_VISIBLE_DEVICES") ? std::getenv("CUDA_VISIBLE_DEVICES") : "";
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        auto next = [&](const char* name) -> const char* {
            if (i + 1 >= argc) { std::fprintf(stderr, "%s needs a value\n", name); std::exit(1); }
            return argv[++i];
        };
        if (a == "--spp") spp = std::atoi(next("--spp"));
        else if (a == "--width") width = std::atoi(next("--width"));
        else if (a == "--height") height = std::atoi(next("--height"));
        else if (a == "--gpus") gpus = std::atoi(next("--gpus"));
        else if (a == "--chunk") chunk = std::atoi(next("--chunk"));
        else if (a == "--seed") seed = std::strtoull(next("--seed"), nullptr, 0);
        else if (a == "--scene-seed") { scene_seed = std::strtoull(next("--scene-seed"), nullptr, 0); have_scene_seed = true; }
        else if (a == "--out") out = next("--out");
        else if (a == "--checkpoint") ckpt_path = next("--checkpoint");
        else if (a == "--checkpoint-every") ckpt_every = std::atoi(next("--checkpoint-every"));
        else if (a == "--resume") resume_path = next("--resume");
        else if (a == "--stop-after-chunks") stop_after = std::atoi(next("--stop-after-chunks"));
        else if (a == "--adaptive") {
            const char* v = next("--adaptive");
            char* end = nullptr;
            adaptive = std::strtod(v, &end);
            if (*end != 0 || !(adaptive >= 0.0)) { std::fprintf(stderr, "--adaptive needs a threshold >= 0\n"); return 1; }
        }
        else if (a == "--min-spp") min_spp = std::atoi(next("--min-spp"));
        else if (a == "--step") step_spp = std::atoi(next("--step"));
        else if (a == "--worker") worker_rank = std::atoi(next("--worker"));
        else if (a == "--shm-fd") shm_fd = std::atoi(next("--shm-fd"));
        else if (a == "--device-list") device_list = next("--device-list");
        else if (scene < 0 && !a.empty() && a[0] != '-') {
            char* end = nullptr;
            long v = std::strtol(a.c_str(), &end, 10);
            if (*end != 0) { std::fprintf(stderr, "Error: There was an error\n"); return 1; }  // parse() failure -> DummyError
            scene = (int)v;
        } else { usage(argv[0]); std::fprintf(stderr, "Error: There was an error\n"); return 1; }
    }
    if (scene < 0) { usage(argv[0]); std::fprintf(stderr, "Error: There was an error\n"); return 1; }
    if (adaptive >= 0.0 && (gpus > 1 || !ckpt_path.empty() || !resume_path.empty())) {
        std::fprintf(stderr, "--adaptive renders on one GPU without checkpoints: it cannot be combined with --gpus > 1, "
                             "--checkpoint or --resume\n");
        return 1;
    }
    if (worker_rank < 0) std::printf("Scene number: %d\n", scene);
    auto t0 = std::chrono::steady_clock::now();
    rtx_scene_defaults def;
    if (rtx_builtin_scene_defaults(scene, &def) != RTX_OK) {
        std::fprintf(stderr, "%s\nError: There was an error\n", rtx_last_error());  // main.rs:179-182
        return 1;
    }
    if (worker_rank < 0) std::printf("Running scene %s\n", def.name);
    if (spp < 0) spp = def.samples;
    if (width < 0) width = def.width;
    if (height < 0) height = def.height;
    if (gpus < 1) gpus = 1;
    if (chunk < 1) chunk = 1;
    if (!have_scene_seed) scene_seed = 0x5254544E57ull + (unsigned long long)scene;
    rtx_scene_desc* desc = nullptr;
    RTX(rtx_builtin_scene(scene, scene_seed, nullptr, &desc));

    if (adaptive >= 0.0) {
        if (min_spp < 0) min_spp = std::max(2, (spp / 64 + 1) / 2 * 2);
        if (step_spp < 0) step_spp = min_spp;
        rtx_ctx* ctx = nullptr;
        rtx_scene* sc = nullptr;
        float *accum = nullptr, *aux = nullptr;
        const size_t bytes = (size_t)width * height * 4 * sizeof(float);
        RTX(rtx_ctx_create(0, nullptr, &ctx));
        RTX(rtx_scene_create(ctx, desc, &sc));
        RTX(rtx_malloc(ctx, bytes, (void**)&accum));
        RTX(rtx_malloc(ctx, bytes, (void**)&aux));
        rtx_render_params p{width, height, 0, spp, def.max_depth, 0, seed};
        rtx_adaptive_params ap{adaptive, min_spp, step_spp};
        rtx_adaptive_stats st{};
        RTX(rtx_render_adaptive(ctx, sc, &p, &ap, accum, aux, &st));
        std::vector<uint8_t> rgba((size_t)width * height * 4);
        RTX(rtx_tonemap_rgba8(ctx, accum, width, height, rgba.data(), 0));
        RTX(rtx_png_write_rgba8(out.c_str(), width, height, rgba.data()));
        std::printf("Adaptive sampling: %lld path samples (%.1f per pixel, at most %d), %d rounds, %d of %d tiles converged, %d at %d spp\n",
                    (long long)st.path_samples, (double)st.path_samples / ((double)width * height), spp, st.rounds,
                    st.tiles_converged, st.tiles, st.tiles_at_max, spp);
        rtx_free(ctx, accum);
        rtx_free(ctx, aux);
        rtx_scene_destroy(sc);
        rtx_ctx_destroy(ctx);
        rtx_scene_desc_free(desc);
        std::printf("%.6fs\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count());
        return 0;
    }

    const bool verbose = std::getenv("RTTNW_VERBOSE") != nullptr;
    auto lap = [&](const char* what) {
        if (verbose) std::fprintf(stderr, "[%8.3f s] %s\n", std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count(), what);
    };
    lap("scene description built");
    const bool static_ranges = !ckpt_path.empty() || !resume_path.empty() || stop_after >= 0;
    const bool one_device_per_process = std::getenv("RTTNW_SINGLE_PROCESS") == nullptr && !(gpus > 1 && static_ranges);
    std::vector<Rank> ranks((size_t)gpus);
    auto worker = [&](int r) {
        Rank& k = ranks[(size_t)r];
        auto chk = [&](int rc) { if (rc != RTX_OK && k.rc == 0) { k.rc = rc; std::fprintf(stderr, "gpu %d: %s\n", r, rtx_last_error()); } return rc == RTX_OK; };
        if (!chk(rtx_ctx_create(one_device_per_process ? 0 : r, nullptr, &k.ctx))) return;
        if (r == 0) lap("context created");
        if (!chk(rtx_scene_create(k.ctx, desc, &k.scene))) return;
        if (r == 0) lap("scene uploaded");
        size_t bytes = (size_t)width * height * 4 * sizeof(float);
        if (!chk(rtx_malloc(k.ctx, bytes, (void**)&k.accum))) return;
        if (!chk(rtx_memset_zero(k.ctx, k.accum, bytes))) return;
        int begin = (int)((long long)r * spp / gpus), end = (int)((long long)(r + 1) * spp / gpus);
        CheckpointHeader hdr;
        std::memset(&hdr, 0, sizeof(hdr));
        std::memcpy(hdr.magic, "RTXACC1", 8);
        hdr.scene = scene; hdr.width = width; hdr.height = height; hdr.spp_total = spp; hdr.gpus = gpus; hdr.rank = r;
        hdr.max_depth = def.max_depth; hdr.seed = seed; hdr.scene_seed = scene_seed;
        std::vector<float> host_acc;
        if (!resume_path.empty()) {
            CheckpointHeader got;
            std::string path = resume_path + "." + std::to_string(r);
            if (!read_checkpoint(path, got, host_acc) || got.scene != scene || got.width != width || got.height != height ||
                got.spp_total != spp || got.gpus != gpus || got.rank != r || got.seed != seed || got.scene_seed != scene_seed ||
                got.max_depth != def.max_depth || got.next_sample < begin || got.next_sample > end) {
                std::fprintf(stderr, "gpu %d: %s is not a checkpoint of this render\n", r, path.c_str());
                k.rc = 1;
                return;
            }
            if (!chk(rtx_memcpy_h2d(k.ctx, k.accum, host_acc.data(), bytes))) return;
            begin = got.next_sample;
        }
        int chunks_done = 0;
        for (int b = begin; b < end; b += chunk) {
            rtx_render_params p;
            std::memset(&p, 0, sizeof(p));
            p.width = width; p.height = height; p.spp_begin = b; p.spp_count = (end - b < chunk) ? end - b : chunk;
            p.max_depth = def.max_depth; p.seed = seed;
            if (!chk(rtx_render(k.ctx, k.scene, &p, k.accum, nullptr))) return;
            ++chunks_done;
            if (!ckpt_path.empty() && (chunks_done % (ckpt_every < 1 ? 1 : ckpt_every) == 0 || b + chunk >= end)) {
                host_acc.resize(bytes / sizeof(float));
                if (!chk(rtx_memcpy_d2h(k.ctx, host_acc.data(), k.accum, bytes))) return;  // ordered after the render on the ctx stream
                hdr.next_sample = b + p.spp_count;
                if (!write_checkpoint(ckpt_path + "." + std::to_string(r), hdr, host_acc)) {
                    std::fprintf(stderr, "gpu %d: cannot write checkpoint %s\n", r, ckpt_path.c_str());
                    k.rc = 1;
                    return;
                }
            }
            if (stop_after >= 0 && chunks_done >= stop_after) { k.rc = 3; return; }  // simulated interruption (tests)
        }
        chk(rtx_ctx_sync(k.ctx));
        if (r == 0) lap("render finished");
    };
    const bool multi_process = gpus > 1 && one_device_per_process;
    std::vector<const float*> peers;
    if (!multi_process && one_device_per_process && worker_rank < 0) see_only_device(device_list, 0);
    if (multi_process || worker_rank >= 0) {
        if (gpus > 16) { std::fprintf(stderr, "at most 16 GPUs\n"); return 1; }
        const size_t frame_bytes = (size_t)width * height * 4 * sizeof(float);
        const size_t shm_bytes = sizeof(SharedFrame) + frame_bytes * (size_t)(gpus - 1);
        const int me = worker_rank >= 0 ? worker_rank : 0;
        if (me == 0) {
            shm_fd = memfd_create("rttnw-frame", 0);  // (no MFD_CLOEXEC: the workers inherit it across exec)
            if (shm_fd < 0 || ftruncate(shm_fd, (off_t)shm_bytes) != 0) { std::perror("memfd_create"); return 1; }
        }
        void* map = mmap(nullptr, shm_bytes, PROT_READ | PROT_WRITE, MAP_SHARED, shm_fd, 0);
        if (map == MAP_FAILED) { std::perror("mmap"); return 1; }
        SharedFrame* sh = (SharedFrame*)map;  // (a fresh memory file is zero-filled: every counter starts at 0)
        float* slots = (float*)((char*)map + sizeof(SharedFrame));
        see_only_device(device_list, me);
        Rank& k = ranks[(size_t)me];
        auto chk = [&](int rc) { if (rc != RTX_OK && k.rc == 0) { k.rc = rc; std::fprintf(stderr, "gpu %d: %s\n", me, rtx_last_error()); } return rc == RTX_OK; };
        auto bring_up = [&]() {
            if (!chk(rtx_ctx_create(0, nullptr, &k.ctx))) return;
            if (me == 0) lap("context created");
            if (!chk(rtx_scene_create(k.ctx, desc, &k.scene))) return;
            if (!chk(rtx_malloc(k.ctx, frame_bytes, (void**)&k.accum))) return;
            if (!chk(rtx_memset_zero(k.ctx, k.accum, frame_bytes))) return;
        };
        // claim chunks of global sample indices until none are left (chunks small enough that the devices finish together)
        const int dyn_chunk = std::max(16, std::min(chunk, spp / (gpus * 6)));
        auto claim_loop = [&]() {
            sh->state[me].store(1);  // from here on the parent waits for this rank
            int mine = 0;
            for (;;) {
                const int b0 = sh->next_sample.fetch_add(dyn_chunk);
                if (b0 >= spp) break;
                rtx_render_params p;
                std::memset(&p, 0, sizeof(p));
                p.width = width; p.height = height; p.spp_begin = b0; p.spp_count = (spp - b0 < dyn_chunk) ? spp - b0 : dyn_chunk;
                p.max_depth = def.max_depth; p.seed = seed;
                if (!chk(rtx_render(k.ctx, k.scene, &p, k.accum, nullptr))) return;
                mine += p.spp_count;
            }
            chk(rtx_ctx_sync(k.ctx));
            sh->samples[me].store(mine);
        };
        if (me != 0) {  // ---- a worker: render what it can claim, leave the accumulator in its slot, end ----
            // CUDA start-ups that overlap slow each other down so that all finish together after ~1.1 s x their number;
            // one after the other each takes ~0.9 s and its device starts rendering right away: wait for the previous
            // rank to be up (or for the frame to be fully claimed, in which case this device is not needed at all)
            while (sh->state[me - 1].load() == 0 && sh->next_sample.load() < spp) usleep(300);
            if (sh->next_sample.load() >= spp) {
                sh->rc[me] = 0;
                sh->state[me].store(2);
                _exit(0);
            }
            bring_up();
            if (k.rc == 0) claim_loop();
            if (k.rc == 0 && sh->samples[me].load() > 0 &&
                rtx_memcpy_d2h(k.ctx, (char*)slots + frame_bytes * (size_t)(me - 1), k.accum, frame_bytes) != RTX_OK) {
                std::fprintf(stderr, "gpu %d: %s\n", me, rtx_last_error());
                k.rc = 1;
            }
            sh->rc[me] = k.rc;
            sh->state[me].store(2);
            _exit(k.rc == 0 ? 0 : 1);  // (no teardown: the process ends here and the driver reclaims the device)
        }
        // ---- the parent: its own device first and alone, then the workers behind it ----
        bring_up();
        if (k.rc != 0) return 1;
        lap("scene uploaded");
        std::vector<pid_t> pids((size_t)gpus, -1);
        std::fflush(stdout);
        std::fflush(stderr);
        for (int r = 1; r < gpus; ++r) {
            pid_t pid = fork();
            if (pid < 0) { std::perror("fork"); break; }
            if (pid == 0) {
                std::vector<std::string> args(argv, argv + argc);
                for (const char* extra : {"--worker", "", "--shm-fd", "", "--device-list", ""}) args.push_back(extra);
                args[args.size() - 5] = std::to_string(r);
                args[args.size() - 3] = std::to_string(shm_fd);
                args[args.size() - 1] = device_list;
                std::vector<char*> cargs;
                for (auto& a : args) cargs.push_back(const_cast<char*>(a.c_str()));
                cargs.push_back(nullptr);
                execv("/proc/self/exe", cargs.data());
                std::perror("execv");
                _exit(127);
            }
            pids[(size_t)r] = pid;
        }
        claim_loop();
        if (k.rc != 0) { for (int r = 1; r < gpus; ++r) if (pids[(size_t)r] > 0) { kill(pids[(size_t)r], SIGKILL); waitpid(pids[(size_t)r], nullptr, 0); } return 1; }
        lap("render finished");
        // every sample index is claimed now. A worker that has not begun to claim can get nothing any more: end it, do
        // not wait for its CUDA start-up; wait for the ones that hold samples.
        int bad = 0, used = 1;
        for (int r = 1; r < gpus; ++r) {
            if (pids[(size_t)r] <= 0) continue;
            if (sh->state[r].load() == 0) {
                kill(pids[(size_t)r], SIGKILL);
                pids[(size_t)r] = -1;  // (not waited for: a process inside the CUDA start-up takes over a second to go; init reaps it)
            } else {
                while (sh->state[r].load() != 2) {
                    int st = 0;
                    if (waitpid(pids[(size_t)r], &st, WNOHANG) == pids[(size_t)r]) {  // died without reporting
                        if (sh->state[r].load() != 2) { std::fprintf(stderr, "gpu %d: worker process died\n", r); bad = 1; }
                        pids[(size_t)r] = -1;
                        break;
                    }
                    usleep(200);
                }
                if (sh->state[r].load() == 2 && sh->rc[r] != 0) bad = 1;
                if (sh->samples[r].load() > 0) ++used;
            }
        }
        if (verbose) {
            std::fprintf(stderr, "           samples per pixel by rank:");
            for (int r = 0; r < gpus; ++r) std::fprintf(stderr, " %d", sh->samples[r].load());
            std::fprintf(stderr, "  (%d of %d devices were up in time)\n", used, gpus);
        }
        if (bad != 0) { for (int r = 1; r < gpus; ++r) if (pids[(size_t)r] > 0) waitpid(pids[(size_t)r], nullptr, 0); return 1; }
        lap("all ranks finished");
        std::vector<void*> staged;
        for (int r = 1; r < gpus; ++r) {
            if (sh->samples[r].load() <= 0) continue;
            void* d = nullptr;
            RTX(rtx_malloc(k.ctx, frame_bytes, &d));
            RTX(rtx_memcpy_h2d(k.ctx, d, (char*)slots + frame_bytes * (size_t)(r - 1), frame_bytes));
            staged.push_back(d);
            peers.push_back((const float*)d);
        }
        std::vector<uint8_t> rgba_mp((size_t)width * height * 4);
        uint8_t* d_rgba_mp = nullptr;
        RTX(rtx_malloc(k.ctx, rgba_mp.size(), (void**)&d_rgba_mp));
        RTX(rtx_reduce_tonemap_peers(k.ctx, k.accum, peers.empty() ? nullptr : peers.data(), (int)peers.size(), width, height, d_rgba_mp));
        RTX(rtx_memcpy_d2h(k.ctx, rgba_mp.data(), d_rgba_mp, rgba_mp.size()));
        lap("frame on the host");
        RTX(rtx_png_write_rgba8(out.c_str(), width, height, rgba_mp.data()));
        lap("png written");
        double secs_mp = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        std::printf("%.6fs\n", secs_mp);  // println!("{:?}", instant.elapsed())
        std::fflush(stdout);
        for (int r = 1; r < gpus; ++r) if (pids[(size_t)r] > 0) waitpid(pids[(size_t)r], nullptr, 0);
        _exit(0);  // like the workers: no context teardown at the end of the process
    }
    std::vector<std::thread> th;
    for (int r = 0; r < gpus; ++r) th.emplace_back(worker, r);
    for (auto& t : th) t.join();
    for (auto& k : ranks) if (k.rc != 0) return k.rc == 3 ? 3 : 1;

    // combine on rank 0: peers' accumulators are read over NVLink by the fused reduce+tonemap kernel
    std::vector<uint8_t> rgba((size_t)width * height * 4);
    uint8_t* d_rgba = nullptr;
    RTX(rtx_malloc(ranks[0].ctx, rgba.size(), (void**)&d_rgba));
    for (int r = 1; r < gpus; ++r) peers.push_back(ranks[(size_t)r].accum);
    RTX(rtx_reduce_tonemap_peers(ranks[0].ctx, ranks[0].accum, peers.empty() ? nullptr : peers.data(), (int)peers.size(), width, height, d_rgba));
    RTX(rtx_memcpy_d2h(ranks[0].ctx, rgba.data(), d_rgba, rgba.size()));
    lap("frame on the host");
    RTX(rtx_png_write_rgba8(out.c_str(), width, height, rgba.data()));  // image::save_buffer("image.png", ..), main.rs:231
    lap("png written");
    rtx_free(ranks[0].ctx, d_rgba);
    for (auto& k : ranks) {
        rtx_free(k.ctx, k.accum);
        rtx_scene_destroy(k.scene);
        rtx_ctx_destroy(k.ctx);
    }
    rtx_scene_desc_free(desc);
    double secs = std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
    std::printf("%.6fs\n", secs);  // println!("{:?}", instant.elapsed())
    return 0;
}
