// waifu2x-b200: command-line driver with the reference's flags, file discovery, model-path and output-naming rules
// (/root/reference/src/main.cpp:17-140 options, :156-160 extensions, :201-209 model path + suffix, :211-274 render loop,
// :275-294 build), over the trt::Img2Img shim (img2img.hpp -> libw2x.so) and the ffmpeg pipes in videoio.hpp.
//
// Differences by design: frames are pipelined (reader thread -> pinned ring -> w2x_submit/w2x_wait -> writer thread: decode, H2D,
// compute, D2H and encode overlap; the reference serialises read -> render -> write on one thread, main.cpp:263-269), `--ffmpegDir` and
// `--modelsDir` are settable (the reference hard-wires "" and "models/"), and a render failure releases the pipes
// before returning -1.  No CLI11/spdlog: the parser below accepts the same spellings and value sets.
//
// Build: make -C waifu2x-tensorrt_b200/csrc cli   (g++ -std=c++17 -pthread, links libw2x.so only)
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <ctime>
#include <filesystem>
#include <functional>
#include <iostream>
#include <map>
#include <memory>
#include <mutex>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "img2img.hpp"
#include "videoio.hpp"

namespace fs = std::filesystem;

namespace {

struct Options {
    std::string model;
    int scale = 0, noise = 0, batchSize = 0, tileSize = 0, deviceId = 0;
    std::vector<int> deviceIds;  // extension: --device 0,1,2,... shards the frames of a render over several GPUs
    trt::Precision precision = trt::Precision::FP16;
    std::string command;  // "render" | "build"
    std::vector<fs::path> inputPaths;
    bool recursive = false, nosuffix = false, tta = false;
    bool alpha = false;  // extension: still images keep their alpha channel (BGRA through Img2Img::renderBgra, PNG out)
    double outputScale = 0;  // extension (> 0 when given): output lround(w F) x lround(h F), at most --scale (Img2Img::submitResized)
    int bitDepth = 8;        // extension: 16 = u16 BGR frames through Img2Img::submitU16, 16-bit PNG stills
    fs::path outputDirectory;
    double blend = 1.0 / 16.0;
    std::string codec = "libx264", pixelFormat = "yuv420p";
    int crf = 23;
    std::string ffmpegDir, modelsDir = "models";
};

struct ParseError : std::runtime_error {
    using std::runtime_error::runtime_error;
};

const char* kUsage =
    "waifu2x-b200\n"
    "Usage: waifu2x-b200 [OPTIONS] SUBCOMMAND\n\n"
    "Options:\n"
    "  -h, --help                    Print this help message and exit\n"
    "  --model TEXT:{cunet/art,swin_unet/art,swin_unet/art_scan,swin_unet/photo} REQUIRED\n"
    "  --scale INT:{1,2,4} REQUIRED  Set the scale factor\n"
    "  --noise INT:{-1,0,1,2,3} REQUIRED\n"
    "  --batchSize INT:POSITIVE REQUIRED\n"
    "  --tileSize INT:{64,128,256,400,640} REQUIRED\n"
    "  --device INT:NONNEGATIVE=0    Set the GPU device ID (extension: a comma-separated list shards frames over several GPUs)\n"
    "  --precision ENUM:{fp16,tf32}=fp16\n"
    "  --modelsDir TEXT=models       Directory holding <model>/[noiseN_][scaleSx].onnx\n\n"
    "Subcommands:\n"
    "  render                        Render image(s)/video(s)\n"
    "    -i, --input PATH ... REQUIRED   --recursive   -o, --output DIR   --nosuffix\n"
    "    --blend FLOAT:{0.125,0.0625,0.03125,0}=0.0625   --tta\n"
    "    --codec TEXT=libx264   --pix_fmt TEXT=yuv420p   --crf INT:[0,51]=23   --ffmpegDir TEXT\n"
    "    --alpha                     Keep the alpha channel of still images (extension; videos are rendered without it)\n"
    "    --outputScale FLOAT:(0,scale]   Output size round(F x input) instead of scale x input: the model's output reduced on the GPU\n"
    "                                by an antialiased bicubic resample (extension; not with --alpha)\n"
    "    --bitDepth INT:{8,16}=8     Bits per channel of the frames the model sees and returns (extension): 16 decodes the input as\n"
    "                                16-bit BGR and writes 16-bit PNG stills; a video keeps --codec / --pix_fmt, so it needs a deep\n"
    "                                --pix_fmt (e.g. yuv420p10le) to keep the bits.  Not with --alpha or --outputScale\n"
    "  build                         Build model\n";

int toInt(const std::string& name, const std::string& v) {
    size_t pos = 0;
    int x = 0;
    try {
        x = std::stoi(v, &pos);
    } catch (...) {
        pos = 0;
    }
    if (pos != v.size() || v.empty()) throw ParseError(name + ": '" + v + "' is not an integer");
    return x;
}

template <class T>
void requireMember(const std::string& name, const T& v, std::initializer_list<T> choices) {
    if (std::find(choices.begin(), choices.end(), v) == choices.end()) throw ParseError(name + ": value not in the allowed set");
}

// Same option spellings, value checks and "required" rules as main.cpp:17-140; options may come before or after the
// subcommand (CLI11 fallthrough), `--opt=value` and `--opt value` both work, -i takes one or more paths.
Options parse(int argc, char** argv) {
    Options o;
    std::set<std::string> seen;
    std::vector<std::string> args(argv + 1, argv + argc);
    for (size_t i = 0; i < args.size(); ++i) {
        std::string a = args[i], inlineVal;
        bool hasInline = false;
        if (a.rfind("--", 0) == 0) {
            const size_t eq = a.find('=');
            if (eq != std::string::npos) { inlineVal = a.substr(eq + 1); a = a.substr(0, eq); hasInline = true; }
        }
        auto value = [&]() -> std::string {
            if (hasInline) return inlineVal;
            if (i + 1 >= args.size()) throw ParseError(a + ": 1 required value missing");
            return args[++i];
        };
        const bool inRender = o.command == "render";
        if (a == "-h" || a == "--help") { std::cout << kUsage; std::exit(0); }
        else if (a == "render" || a == "build") {
            if (!o.command.empty()) throw ParseError("exactly one subcommand is required");
            o.command = a;
        }
        else if (a == "--model") { o.model = value(); requireMember<std::string>(a, o.model, {"cunet/art", "swin_unet/art", "swin_unet/art_scan", "swin_unet/photo"}); }
        else if (a == "--scale") { o.scale = toInt(a, value()); requireMember(a, o.scale, {1, 2, 4}); }
        else if (a == "--noise") { o.noise = toInt(a, value()); requireMember(a, o.noise, {-1, 0, 1, 2, 3}); }
        else if (a == "--batchSize") { o.batchSize = toInt(a, value()); if (o.batchSize <= 0) throw ParseError(a + ": must be positive"); }
        else if (a == "--tileSize") { o.tileSize = toInt(a, value()); requireMember(a, o.tileSize, {64, 128, 256, 400, 640}); }
        else if (a == "--device") {
            // the reference takes one id (main.cpp:70-74); a comma-separated list renders frame f on the (f mod n)-th listed GPU
            std::string list = value();
            o.deviceIds.clear();
            size_t pos = 0;
            while (pos <= list.size()) {
                const size_t comma = std::min(list.find(',', pos), list.size());
                const int id = toInt(a, list.substr(pos, comma - pos));
                if (id < 0) throw ParseError(a + ": must be non-negative");
                o.deviceIds.push_back(id);
                pos = comma + 1;
            }
            o.deviceId = o.deviceIds.front();
        }
        else if (a == "--precision") {
            std::string v = value();
            std::transform(v.begin(), v.end(), v.begin(), ::tolower);
            if (v == "fp16") o.precision = trt::Precision::FP16;
            else if (v == "tf32") o.precision = trt::Precision::TF32;
            else throw ParseError(a + ": expected fp16 or tf32");
        }
        else if (a == "--modelsDir") o.modelsDir = value();
        else if (inRender && (a == "-i" || a == "--input")) {
            if (hasInline) o.inputPaths.emplace_back(inlineVal);
            while (i + 1 < args.size() && args[i + 1].rfind("-", 0) != 0 && args[i + 1] != "build") o.inputPaths.emplace_back(args[++i]);
            for (const auto& p : o.inputPaths)
                if (!fs::exists(p)) throw ParseError(a + ": Path does not exist: " + p.string());
        }
        else if (inRender && a == "--recursive") o.recursive = true;
        else if (inRender && (a == "-o" || a == "--output")) {
            o.outputDirectory = value();
            if (!fs::is_directory(o.outputDirectory)) throw ParseError(a + ": Directory does not exist: " + o.outputDirectory.string());
        }
        else if (inRender && a == "--nosuffix") o.nosuffix = true;
        else if (inRender && a == "--blend") {
            const std::string v = value();
            try { o.blend = std::stod(v); } catch (...) { throw ParseError(a + ": '" + v + "' is not a number"); }
            requireMember(a, o.blend, {1.0 / 8.0, 1.0 / 16.0, 1.0 / 32.0, 0.0});
        }
        else if (inRender && a == "--tta") o.tta = true;
        else if (inRender && a == "--alpha") o.alpha = true;
        else if (inRender && a == "--outputScale") {
            const std::string v = value();
            size_t pos = 0;
            try { o.outputScale = std::stod(v, &pos); } catch (...) { pos = 0; }
            if (v.empty() || pos != v.size() || !std::isfinite(o.outputScale)) throw ParseError(a + ": '" + v + "' is not a number");
            if (o.outputScale <= 0) throw ParseError(a + ": must be positive");
        }
        else if (a == "--bitDepth") { o.bitDepth = toInt(a, value()); requireMember(a, o.bitDepth, {8, 16}); }
        else if (inRender && a == "--codec") o.codec = value();
        else if (inRender && a == "--pix_fmt") o.pixelFormat = value();
        else if (inRender && a == "--crf") { o.crf = toInt(a, value()); if (o.crf < 0 || o.crf > 51) throw ParseError(a + ": value not in range 0 to 51"); }
        else if (inRender && a == "--ffmpegDir") o.ffmpegDir = value();
        else throw ParseError("The following argument was not expected: " + args[i]);
        seen.insert(a == "-i" ? "--input" : a);
    }
    for (const char* req : {"--model", "--scale", "--noise", "--batchSize", "--tileSize"})
        if (!seen.count(req)) throw ParseError(std::string(req) + " is required");
    if (o.command.empty()) throw ParseError("A subcommand is required");
    if (o.command == "render" && o.inputPaths.empty()) throw ParseError("--input is required");
    if (o.outputScale > o.scale) throw ParseError("--outputScale: at most --scale (" + std::to_string(o.scale) + "); the resample only reduces the model's output");
    if (o.outputScale > 0 && o.alpha) throw ParseError("--outputScale: not available with --alpha");
    if (seen.count("--bitDepth") && o.command != "render") throw ParseError("--bitDepth: applies to render only");
    if (o.bitDepth == 16 && o.alpha) throw ParseError("--bitDepth: 16 is not available with --alpha");
    if (o.bitDepth == 16 && o.outputScale > 0) throw ParseError("--bitDepth: 16 is not available with --outputScale");
    return o;
}

// utilities/path.h:8-37: explicit files and directory entries whose extension is in the list; order of discovery
std::vector<fs::path> findFilesByExtension(const std::vector<fs::path>& paths, const std::vector<std::string>& exts, bool recursive) {
    std::vector<fs::path> out;
    auto consider = [&](const fs::path& p) {
        if (p.has_extension() && std::find(exts.begin(), exts.end(), p.extension().string()) != exts.end()) out.push_back(p);
    };
    for (const auto& p : paths) {
        if (fs::is_regular_file(p)) consider(p);
        else if (fs::is_directory(p)) {
            if (recursive) for (const auto& e : fs::recursive_directory_iterator(p)) consider(e.path());
            else for (const auto& e : fs::directory_iterator(p)) consider(e.path());
        }
    }
    return out;
}

// "[HH:MM:SS.mmm] [LEVEL] text" (main.cpp:9,15)
void logLine(trt::Severity sev, const std::string& msg) {
    static const char* names[] = {"FATAL", "ERROR", "WARN ", "INFO ", "DEBUG", "TRACE"};
    if (sev > trt::Severity::info) return;  // console level info (main.cpp:14)
    const auto now = std::chrono::system_clock::now();
    const std::time_t t = std::chrono::system_clock::to_time_t(now);
    const int ms = (int)(std::chrono::duration_cast<std::chrono::milliseconds>(now.time_since_epoch()).count() % 1000);
    std::tm tm{};
    localtime_r(&t, &tm);
    std::printf("[%02d:%02d:%02d.%03d] [%s] %s\n", tm.tm_hour, tm.tm_min, tm.tm_sec, ms, names[(int)sev], msg.c_str());
    std::fflush(stdout);
}

struct PinnedBuffer {  // page-locked so the copy engines stream at full rate while the pipes block on ffmpeg
    unsigned char* p = nullptr;
    size_t cap = 0;
    void reserve(size_t n) {
        if (n <= cap) return;
        if (p) w2x_host_free(p);
        p = static_cast<unsigned char*>(w2x_host_alloc(n));
        if (!p) throw std::runtime_error("could not allocate pinned host memory");
        cap = n;
    }
    ~PinnedBuffer() { if (p) w2x_host_free(p); }
};

}  // namespace

int main(int argc, char* argv[]) {
    Options o;
    try {
        o = parse(argc, argv);
        if (o.model == "cunet/art" && o.scale == 4) throw std::runtime_error("cunet/art does not support scale factor 4.");
        if (o.noise == -1 && o.scale == 1) throw std::runtime_error("Noise level -1 does not support scale factor 1.");
    } catch (const ParseError& e) {
        std::cerr << e.what() << "\nRun with --help for more information.\n";
        return 106;
    } catch (const std::exception& e) {
        std::cerr << e.what();
        return -1;
    }

    const std::vector<std::string> extensions = {".png", ".jpg", ".jpeg", ".bmp", ".tif", ".tiff", ".mp4", ".avi", ".mkv"};
    auto files = findFilesByExtension(o.inputPaths, extensions, o.recursive);

    size_t fileIndex = 0, frameIndex = 0, frameCount = 0;
    const size_t fileCount = files.size();
    trt::Img2Img engine;
    engine.setMessageCallback(logLine);
    engine.setProgressCallback([&](int current, int total, double speed) {
        char line[256];
        std::snprintf(line, sizeof(line), "Rendered file %zu/%zu, frame %zu/%zu, batch %d/%d @ %.2f it/s", fileIndex, fileCount, frameIndex,
                      frameCount, current, total, speed);
        logLine(trt::Severity::info, line);
    });

    const std::string noiseTag = o.noise == -1 ? "" : "noise" + std::to_string(o.noise);
    const std::string scaleTag = o.scale == 1 ? "" : "scale" + std::to_string(o.scale);
    std::string modelPath = o.modelsDir + "/" + o.model + "/" + (noiseTag.empty() ? "" : noiseTag + "_") + (scaleTag.empty() ? "" : scaleTag + "x") + ".onnx";
    // main.cpp:201-204 yields "noiseN_.onnx" (trailing underscore) for scale 1; the released archives name that file "noiseN.onnx"
    if (scaleTag.empty() && !noiseTag.empty() && !fs::exists(modelPath)) {
        const std::string alt = o.modelsDir + "/" + o.model + "/" + noiseTag + ".onnx";
        if (fs::exists(alt)) modelPath = alt;
    }
    std::string flatModel = o.model;
    std::replace(flatModel.begin(), flatModel.end(), '/', '_');
    const std::string suffix = "(" + flatModel + ")" + (noiseTag.empty() ? "" : "(" + noiseTag + ")") + (scaleTag.empty() ? "" : "(" + scaleTag + ")") + (o.tta ? "(tta)" : "");

    if (o.command == "build") {
        trt::BuildConfig c;
        c.deviceId = o.deviceId;
        c.precision = o.precision;
        c.minBatchSize = c.optBatchSize = c.maxBatchSize = o.batchSize;
        c.minChannels = c.optChannels = c.maxChannels = 3;
        c.minWidth = c.optWidth = c.maxWidth = c.minHeight = c.optHeight = c.maxHeight = o.tileSize;
        return engine.build(modelPath, c) ? 0 : -1;
    }

    trt::RenderConfig rc;
    rc.deviceId = o.deviceId;
    rc.precision = o.precision;
    rc.batchSize = o.batchSize;
    rc.channels = 3;
    rc.height = rc.width = o.tileSize;
    rc.scaling = o.scale;
    rc.overlap = {o.blend, o.blend};
    rc.tta = o.tta;
    std::unique_ptr<trt::Img2ImgPool> pool;
    if (o.deviceIds.size() > 1) {
        pool = std::make_unique<trt::Img2ImgPool>(o.deviceIds);
        if (!pool->valid()) { logLine(trt::Severity::error, "could not create the engine pool for --device list"); return -1; }
        pool->setMessageCallback(logLine);
        if (!pool->load(modelPath, rc)) return -1;
    } else if (!engine.load(modelPath, rc)) {
        return -1;
    }
    const bool deep = o.bitDepth == 16;
    auto submitFrame = [&](const unsigned char* src, int w, int h, size_t ss, unsigned char* dst, const FrameSize& ds) {
        if (deep) {
            const auto* s16 = reinterpret_cast<const uint16_t*>(src);
            auto* d16 = reinterpret_cast<uint16_t*>(dst);
            return pool ? pool->submitU16(s16, w, h, ss, d16, (size_t)ds.width * 6) : engine.submitU16(s16, w, h, ss, d16, (size_t)ds.width * 6);
        }
        if (o.outputScale > 0)
            return pool ? pool->submitResized(src, w, h, ss, dst, ds.width, ds.height, (size_t)ds.width * 3)
                        : engine.submitResized(src, w, h, ss, dst, ds.width, ds.height, (size_t)ds.width * 3);
        return pool ? pool->submit(src, w, h, ss, dst, (size_t)ds.width * 3) : engine.submit(src, w, h, ss, dst, (size_t)ds.width * 3);
    };
    auto waitFrame = [&](int ticket) { return pool ? pool->wait(ticket) : engine.wait(ticket); };

    // Decode, GPU and encode are decoupled (SURVEY 8f rank 1; the reference serialises them on one thread, main.cpp:263-269):
    // a reader thread fills a ring of pinned input frames from the ffmpeg pipe, this thread submits them to the engine (at most
    // three in flight, Engine::kSlots) and retires them in order, a writer thread drains finished frames into the encoder pipe.
    const int nDev = (int)std::max<size_t>(o.deviceIds.size(), 1);
    const int kInFlight = 3 * nDev, kRing = kInFlight + 3;  // three frames in flight per GPU + slack for the reader / writer threads
    enum SlotState { FREE, FILLED, SUBMITTED, DONE };
    std::vector<PinnedBuffer> in(kRing), out(kRing);
    VideoCapture capture;
    VideoWriter writer;
    capture.setFfmpegDir(o.ffmpegDir).setBitDepth(o.bitDepth);
    writer.setFfmpegDir(o.ffmpegDir).setConstantRateFactor(o.crf).setBitDepth(o.bitDepth);
    try {
        for (auto& file : files) {
            capture.setChannels(3).open(file.string());
            // --alpha: a still image is decoded again as BGRA (the frame count is known once ffprobe has run)
            const bool bgra = o.alpha && capture.getFrameCount() == 1;
            if (bgra) capture.setChannels(4).open(file.string());
            else if (o.alpha) logLine(trt::Severity::warn, "--alpha applies to still images; " + file.string() + " is rendered without alpha");
            const FrameSize inSize = capture.getFrameSize();
            FrameSize outSize = inSize * o.scale;
            std::string sizeTag;
            if (o.outputScale > 0) {
                outSize = {std::max(1, (int)std::lround(inSize.width * o.outputScale)), std::max(1, (int)std::lround(inSize.height * o.outputScale))};
                sizeTag = "(" + std::to_string(outSize.width) + "x" + std::to_string(outSize.height) + ")";
            }
            frameIndex = 0;
            frameCount = (size_t)capture.getFrameCount();
            if (!o.outputDirectory.empty()) file = o.outputDirectory / file.filename();
            if (!o.nosuffix) file.replace_filename(file.stem().string() + suffix + sizeTag + file.extension().string());
            if (frameCount == 1) {
                file.replace_extension(".png");
                writer.setFrameRate(1).setPixelFormat(deep ? "rgb48be" : "").setCodec("");   // 16-bit: a 16-bit PNG
            } else {
                file.replace_extension(".mp4");
                writer.setFrameRate(capture.getFrameRate()).setPixelFormat(o.pixelFormat).setCodec(o.codec);
            }
            writer.setFrameSize(outSize).setOutputFile(file.string()).setChannels(bgra ? 4 : 3);
            writer.open();
            if (bgra) {  // one frame, synchronously; with a --device list on the pool's first engine
                in[0].reserve(inSize.bytes(4));
                out[0].reserve(outSize.bytes(4));
                if (!capture.read(in[0].p)) throw std::runtime_error("could not read \"" + file.string() + "\"");
                w2x_engine* e = pool ? pool->engine(0) : engine.handle();
                if (!w2x_render_bgra(e, in[0].p, inSize.width, inSize.height, (size_t)inSize.width * 4, out[0].p, (size_t)outSize.width * 4))
                    throw std::runtime_error("render failed");
                frameIndex = 1;
                writer.write(out[0].p, outSize);
                capture.release();
                writer.release();
                if (writer.exitStatus() != 0) throw std::runtime_error("ffmpeg failed to encode \"" + file.string() + "\" (exit status " + std::to_string(writer.exitStatus()) + ")");
                fileIndex++;
                continue;
            }
            for (int s = 0; s < kRing; ++s) { in[s].reserve(inSize.bytes(3, o.bitDepth)); out[s].reserve(outSize.bytes(3, o.bitDepth)); }

            std::mutex mu;
            std::condition_variable cv;
            std::vector<SlotState> state(kRing, FREE);
            size_t framesRead = frameCount;  // lowered by the reader if the pipe ends early
            bool abort = false;
            std::exception_ptr failure;
            auto fail = [&](std::exception_ptr e) {
                std::lock_guard<std::mutex> lk(mu);
                if (!failure) failure = e;
                abort = true;
                cv.notify_all();
            };
            auto waitFor = [&](size_t f, SlotState want) {  // true when slot f % kRing reached `want`; false on abort / end of input
                std::unique_lock<std::mutex> lk(mu);
                cv.wait(lk, [&] { return abort || state[f % kRing] == want || (want == FILLED && f >= framesRead); });
                return !abort && state[f % kRing] == want && f < framesRead;
            };
            auto setState = [&](size_t f, SlotState st) {
                std::lock_guard<std::mutex> lk(mu);
                state[f % kRing] = st;
                cv.notify_all();
            };
            std::thread reader([&] {
                try {
                    for (size_t f = 0; f < frameCount; ++f) {
                        if (!waitFor(f, FREE)) return;
                        if (!capture.read(in[f % kRing].p)) {
                            std::lock_guard<std::mutex> lk(mu);
                            framesRead = f;
                            cv.notify_all();
                            return;
                        }
                        setState(f, FILLED);
                    }
                } catch (...) { fail(std::current_exception()); }
            });
            std::thread sink([&] {
                try {
                    for (size_t f = 0; f < frameCount; ++f) {
                        {
                            std::unique_lock<std::mutex> lk(mu);
                            cv.wait(lk, [&] { return abort || state[f % kRing] == DONE || f >= framesRead; });
                            if (abort || f >= framesRead) return;
                        }
                        writer.write(out[f % kRing].p, outSize);
                        setState(f, FREE);
                    }
                } catch (...) { fail(std::current_exception()); }
            });
            std::vector<int> tickets(kRing);
            size_t submitted = 0, retired = 0;
            auto retire = [&]() {
                if (!waitFrame(tickets[retired % kRing])) throw std::runtime_error("render failed");
                setState(retired, DONE);
                ++retired;
                frameIndex++;
            };
            try {
                while (waitFor(submitted, FILLED)) {
                    if (submitted - retired >= (size_t)kInFlight) retire();
                    const int s = (int)(submitted % kRing);
                    tickets[s] = submitFrame(in[s].p, inSize.width, inSize.height, (size_t)inSize.width * 3 * (o.bitDepth / 8), out[s].p, outSize);
                    if (tickets[s] < 0) throw std::runtime_error("render failed");
                    setState(submitted, SUBMITTED);
                    ++submitted;
                }
                while (retired < submitted) retire();
            } catch (...) { fail(std::current_exception()); }
            reader.join();
            sink.join();
            if (failure) std::rethrow_exception(failure);
            capture.release();
            writer.release();
            if (writer.exitStatus() != 0) throw std::runtime_error("ffmpeg failed to encode \"" + file.string() + "\" (exit status " + std::to_string(writer.exitStatus()) + ")");
            fileIndex++;
        }
    } catch (const std::exception& e) {
        logLine(trt::Severity::error, e.what());
        capture.release();
        writer.release();
        return -1;
    }
    return 0;
}
