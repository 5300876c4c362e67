// Frame feed / sink over ffprobe + ffmpeg child processes (raw bgr24 over popen pipes): header-only re-creation of the
// reference's VideoCapture (/root/reference/src/videoio/capture.{h,cpp}) and VideoWriter (writer.{h,cpp}) with the same
// class names, method names, command lines (capture.cpp:65-68,96-99; writer.cpp:24-33) and error behaviour (std::exception
// on failure), minus OpenCV: frames are raw BGR8 HWC buffers (cv::Mat overloads appear when <opencv2/core.hpp> was included).
// setChannels(4) on either class switches the raw frames to BGRA8 (`-pix_fmt bgra` instead of `bgr24`, nothing else changes), and
// setBitDepth(16) to native-endian u16 BGR (`-pix_fmt bgr48le`; 16-bit BGRA is refused).
//
// Fixes relative to the reference (SURVEY 8f rank 1): the command prefix (`ffmpegDir`) is settable on BOTH classes and is
// honoured by VideoWriter::open (the reference ignores it, writer.cpp:24); release() uses pclose on every platform (the
// reference calls _pclose unconditionally, capture.cpp:132, which does not build on Linux, README.md:95).
#pragma once
#include <algorithm>
#include <cstdint>
#include <cstdio>
#include <filesystem>
#include <map>
#include <sstream>
#include <stdexcept>
#include <string>
#if defined(__linux__)
#include <fcntl.h>
#endif

// 1 MiB kernel pipe buffers (Linux default is 64 KiB): a 4K bgr24 frame is 24.9 MB, so fewer, larger transfers per frame
inline void growPipe(FILE* p) {
#if defined(__linux__) && defined(F_SETPIPE_SZ)
    if (p) (void)fcntl(fileno(p), F_SETPIPE_SZ, 1 << 20);
#else
    (void)p;
#endif
}

struct FrameSize {  // stands in for cv::Size2i
    int width = -1, height = -1;
    bool operator==(const FrameSize& o) const { return width == o.width && height == o.height; }
    bool operator!=(const FrameSize& o) const { return !(*this == o); }
    FrameSize operator*(int s) const { return {width * s, height * s}; }
    size_t bytes(int channels = 3, int bitDepth = 8) const { return (size_t)width * height * channels * (bitDepth / 8); }
};

// A path inside the double quotes of the reference's command lines (capture.cpp:65-68,96-99; writer.cpp:24-33).  The reference pastes
// the raw path, so a file name containing " $ ` or \ would be interpreted by the shell (the CLI feeds this from recursive directory
// discovery, i.e. untrusted names); those four characters are backslash-escaped, every other path yields the reference's exact text.
inline std::string quotedPath(const std::string& path) {
    std::string q = "\"";
    for (char c : path) {
        if (c == '"' || c == '$' || c == '`' || c == '\\') q += '\\';
        q += c;
    }
    return q + "\"";
}

// ffmpeg's name of the raw frame layout with `channels` samples of `bitDepth` bits per pixel
inline const char* rawPixelFormat(int channels, int bitDepth = 8) {
    if (bitDepth != 8 && bitDepth != 16) throw std::invalid_argument("bit depth must be 8 or 16");
    if (channels != 3 && channels != 4) throw std::invalid_argument("channels must be 3 or 4");
    if (bitDepth == 16) {
        if (channels == 4) throw std::invalid_argument("16-bit frames have 3 channels");
        return "bgr48le";
    }
    return channels == 3 ? "bgr24" : "bgra";
}

class VideoCapture {
public:
    VideoCapture() noexcept = default;
    virtual ~VideoCapture() { release(); }
    VideoCapture(const VideoCapture&) = delete;
    VideoCapture& operator=(const VideoCapture&) = delete;

    // capture.cpp:57-111
    void open(const std::string& path) {
        release();
        try {
            if (!std::filesystem::exists(path)) throw std::runtime_error("input file does not exist");
            const std::string probe = ffmpegDir + "ffprobe -v error -select_streams v:0 -show_entries "
                                      "stream=width,height,r_frame_rate,nb_frames -of default=noprint_wrappers=1 " + quotedPath(path);
            FILE* p = popen(probe.c_str(), "r");
            if (!p) throw std::runtime_error("could not open ffprobe with command\"" + probe + "\"");
            char buffer[128];
            std::string output;
            while (fgets(buffer, sizeof(buffer), p) != nullptr) output += buffer;
            pclose(p);
            std::transform(output.begin(), output.end(), output.begin(), ::tolower);
            if (output.find("invalid") != std::string::npos) throw std::runtime_error("input file is invalid");
            const auto props = parseKeyValues(output);
            frameSize.width = std::stoi(props.at("width"));
            frameSize.height = std::stoi(props.at("height"));
            frameRate = fraction(props.at("r_frame_rate"));
            frameCount = props.at("nb_frames") == "n/a" ? 1 : std::stoi(props.at("nb_frames"));  // no frame count => an image
            const std::string cmd = ffmpegDir + "ffmpeg -v error -i " + quotedPath(path) + " -f image2pipe -vcodec rawvideo -pix_fmt " + rawPixelFormat(channels, bitDepth) + " -";
            pipe = popen(cmd.c_str(), "r");
            if (!pipe) throw std::runtime_error("could not open ffmpeg with command\"" + cmd + "\"");
            growPipe(pipe);
            opened = true;
            frameIndex = -1;
        } catch (...) {
            release();
            throw;
        }
    }

    [[nodiscard]] bool isOpened() const noexcept { return opened; }

    // capture.cpp:116-128: one blocking read of W*H*channels*bitDepth/8 bytes; false after the last frame
    bool read(uint8_t* bgr) {
        if (!opened) throw std::runtime_error("video capture is not opened");
        if (frameIndex + 1 >= frameCount) return false;
        const size_t want = frameSize.bytes(channels, bitDepth);
        size_t got = 0;
        while (got < want) {
            const size_t n = fread(bgr + got, 1, want - got, pipe);
            if (n == 0) break;
            got += n;
        }
        if (got != want) throw std::runtime_error("could not read frame from pipe");
        ++frameIndex;
        return true;
    }
#ifdef OPENCV_CORE_HPP
    bool read(cv::Mat& frame) {
        frame.create(frameSize.height, frameSize.width, CV_8UC3);
        return read(frame.data);
    }
#endif

    void release() {
        if (pipe) pclose(pipe);
        pipe = nullptr;
        opened = false;
    }

    [[nodiscard]] const std::string& getFfmpegDir() const noexcept { return ffmpegDir; }
    VideoCapture& setFfmpegDir(const std::string& value) { ffmpegDir = value; return *this; }  // missing in the reference (capture.h)
    // 3 (BGR, the default) or 4 (BGRA); applies from the next open()
    VideoCapture& setChannels(int value) { rawPixelFormat(value, bitDepth); channels = value; return *this; }
    [[nodiscard]] int getChannels() const noexcept { return channels; }
    // 8 (the default) or 16 (3 channels only); applies from the next open()
    VideoCapture& setBitDepth(int value) { rawPixelFormat(channels, value); bitDepth = value; return *this; }
    [[nodiscard]] int getBitDepth() const noexcept { return bitDepth; }
    [[nodiscard]] const FrameSize& getFrameSize() const noexcept { return frameSize; }
    [[nodiscard]] double getFrameRate() const noexcept { return frameRate; }
    [[nodiscard]] int getFrameCount() const noexcept { return frameCount; }
    [[nodiscard]] int getFrameIndex() const noexcept { return frameIndex; }

private:
    static std::map<std::string, std::string> parseKeyValues(const std::string& text) {
        std::map<std::string, std::string> m;
        std::istringstream in(text);
        std::string line;
        while (std::getline(in, line)) {
            while (!line.empty() && (line.back() == '\r' || line.back() == ' ')) line.pop_back();
            const size_t eq = line.find('=');
            if (eq != std::string::npos) m[line.substr(0, eq)] = line.substr(eq + 1);
        }
        return m;
    }
    static double fraction(const std::string& s) {
        const size_t slash = s.find('/');
        if (slash == std::string::npos) return std::stod(s);
        const double den = std::stod(s.substr(slash + 1));
        return den == 0 ? 0.0 : std::stod(s.substr(0, slash)) / den;
    }

    FILE* pipe = nullptr;
    bool opened = false;
    std::string ffmpegDir;
    FrameSize frameSize;
    double frameRate = -1;
    int frameCount = -1;
    int frameIndex = -1;
    int channels = 3;
    int bitDepth = 8;
};

class VideoWriter {
public:
    VideoWriter() noexcept = default;
    virtual ~VideoWriter() noexcept { release(); }
    VideoWriter(const VideoWriter&) = delete;
    VideoWriter& operator=(const VideoWriter&) = delete;

    // writer.cpp:15-40
    void open() {
        release();
        if (frameSize.width <= 0 || frameSize.height <= 0) throw std::invalid_argument("frame size must be greater than 0");
        if (outputFile.empty()) throw std::invalid_argument("output file is empty");
        const std::string cmd = ffmpegDir + "ffmpeg -v error -y -f rawvideo -vcodec rawvideo -s " + std::to_string(frameSize.width) + "x" +
                                std::to_string(frameSize.height) + " -pix_fmt " + rawPixelFormat(channels, bitDepth) + (frameRate <= 0 ? "" : " -r " + std::to_string(frameRate)) +
                                " -i -" + (codec.empty() ? "" : " -vcodec " + codec) + (pixelFormat.empty() ? "" : " -pix_fmt " + pixelFormat) +
                                (crf < 0 ? "" : " -crf " + std::to_string(crf)) + (quality < 0 ? "" : " -q:v " + std::to_string(quality)) +
                                " " + quotedPath(outputFile);
        pipe = popen(cmd.c_str(), "w");
        if (!pipe) throw std::runtime_error("could not open ffmpeg pipe");
        growPipe(pipe);
        opened = true;
    }

    [[nodiscard]] bool isOpened() const noexcept { return opened; }

    // writer.cpp:45-57
    void write(const uint8_t* bgr, const FrameSize& size) {
        if (!opened) throw std::runtime_error("video writer is not opened");
        if (size != frameSize) throw std::invalid_argument("frame size does not match");
        const size_t n = frameSize.bytes(channels, bitDepth);
        if (fwrite(bgr, 1, n, pipe) != n) throw std::runtime_error("could not write frame to pipe");
    }
#ifdef OPENCV_CORE_HPP
    void write(const cv::Mat& frame) {
        if (frame.type() != CV_8UC3) throw std::invalid_argument("frame type must be CV_8UC3");
        write(frame.data, FrameSize{frame.cols, frame.rows});
    }
#endif

    // Closes the encoder pipe; the exit status of ffmpeg is kept (the reference drops it, writer.cpp:59-66): a failed encode must
    // not look like success to the caller.
    void release() noexcept {
        if (pipe) lastStatus = pclose(pipe);
        pipe = nullptr;
        opened = false;
    }
    // 0 when the last closed encoder exited cleanly (or none was opened)
    [[nodiscard]] int exitStatus() const noexcept { return lastStatus; }

    [[nodiscard]] const std::string& getFfmpegDir() const noexcept { return ffmpegDir; }
    [[nodiscard]] const FrameSize& getFrameSize() const noexcept { return frameSize; }
    [[nodiscard]] double getFrameRate() const noexcept { return frameRate; }
    [[nodiscard]] const std::string& getOutputFile() const noexcept { return outputFile; }
    [[nodiscard]] const std::string& getPixelFormat() const noexcept { return pixelFormat; }
    [[nodiscard]] const std::string& getCodec() const noexcept { return codec; }
    [[nodiscard]] int getConstantRateFactor() const noexcept { return crf; }
    [[nodiscard]] int getQuality() const noexcept { return quality; }

    // fluent setters that throw while the writer is open (writer.cpp:102-166)
    VideoWriter& setFfmpegDir(const std::string& v) { guard(); ffmpegDir = v; return *this; }
    VideoWriter& setFrameSize(const FrameSize& v) { guard(); frameSize = v; return *this; }
    VideoWriter& setFrameRate(double v) { guard(); frameRate = v; return *this; }
    VideoWriter& setOutputFile(const std::string& v) { guard(); outputFile = v; return *this; }
    VideoWriter& setPixelFormat(const std::string& v) { guard(); pixelFormat = v; return *this; }
    VideoWriter& setCodec(const std::string& v) { guard(); codec = v; return *this; }
    VideoWriter& setConstantRateFactor(int v) { guard(); crf = v; return *this; }
    VideoWriter& setQuality(int v) { guard(); quality = v; return *this; }
    // 3 (BGR, the default) or 4 (BGRA): the layout of the frames given to write()
    VideoWriter& setChannels(int v) { guard(); rawPixelFormat(v, bitDepth); channels = v; return *this; }
    [[nodiscard]] int getChannels() const noexcept { return channels; }
    // 8 (the default) or 16 (3 channels only): the sample size of the frames given to write()
    VideoWriter& setBitDepth(int v) { guard(); rawPixelFormat(channels, v); bitDepth = v; return *this; }
    [[nodiscard]] int getBitDepth() const noexcept { return bitDepth; }

private:
    void guard() const {
        if (opened) throw std::runtime_error("cannot change a video writer property while it is open");
    }
    FILE* pipe = nullptr;
    bool opened = false;
    std::string ffmpegDir;
    FrameSize frameSize;
    double frameRate = -1;
    std::string outputFile, pixelFormat, codec;
    int crf = -1, quality = -1;
    int lastStatus = 0;
    int channels = 3;
    int bitDepth = 8;
};
