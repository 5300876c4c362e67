#include "hostutil.h"

#include <cctype>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <algorithm>
#include <filesystem>
#include <fstream>
#include <sstream>

namespace w2x {

// ------------------------------------------------------------------------------------------------
// Tile grid.  Same integer results as calculateTiles (img2img_render.cpp:7-66): std::lround is
// half-away-from-zero; the reference uses inputTileSize.width for both dims of the scaled output tile
// (:11-14); tiles are enumerated x-outer / y-inner (:43-44).
// ------------------------------------------------------------------------------------------------
TileGrid calculateTiles(int inW, int inH, int outW, int outH, int tileW, int tileH, int outTileW, int outTileH,
                        int scaling, double overlapX, double overlapY) {
    if (tileW <= 0 || tileH <= 0 || outTileW <= 0 || outTileH <= 0 || scaling <= 0 || inW <= 0 || inH <= 0)
        throw Error("calculateTiles: invalid sizes");
    TileGrid g;
    const int sotW = tileW * scaling, sotH = tileW * scaling;  // sic
    g.scaledInW = (int)std::lround((double)outTileW / sotW * tileW);
    g.scaledInH = (int)std::lround((double)outTileH / sotH * tileH);
    g.inOvX = (int)std::lround(tileW * overlapX);
    g.inOvY = (int)std::lround(tileH * overlapY);
    g.outOvX = (int)std::lround(sotW * overlapX);
    g.outOvY = (int)std::lround(sotH * overlapY);
    if (g.scaledInW - g.inOvX <= 0 || g.scaledInH - g.inOvY <= 0) throw Error("calculateTiles: overlap too large");
    g.nx = (int)std::lround(std::ceil((double)(inW - g.inOvX) / (g.scaledInW - g.inOvX)));
    g.ny = (int)std::lround(std::ceil((double)(inH - g.inOvY) / (g.scaledInH - g.inOvY)));
    // A frame no larger than the input overlap makes tiling.x / tiling.y non-positive: the reference's loops (:43-44) then emit no
    // rects while its tileCount = x * y can even come out positive (both negative) and index past the empty vectors.  Report an
    // empty grid instead, so that every caller's `count <= 0` guard fires.
    g.count = (g.nx < 1 || g.ny < 1) ? 0 : g.nx * g.ny;
    g.inRects.reserve(g.count > 0 ? g.count : 0);
    g.outRects.reserve(g.count > 0 ? g.count : 0);
    const int bx = (tileW - g.scaledInW) / 2, by = (tileH - g.scaledInH) / 2;  // C++ truncating division
    for (int i = 0; i < g.nx; ++i) {
        for (int j = 0; j < g.ny; ++j) {
            g.inRects.push_back({-bx + i * g.scaledInW - i * g.inOvX, -by + j * g.scaledInH - j * g.inOvY, tileW, tileH});
            const int x = i * outTileW - i * g.outOvX;
            const int y = j * outTileH - j * g.outOvY;
            g.outRects.push_back({x, y, x + outTileW > outW ? outW - x : outTileW,
                                  y + outTileH > outH ? outH - y : outTileH});
        }
    }
    return g;
}

std::vector<float> blendRamp(int overlap) {
    std::vector<float> r((size_t)(overlap > 0 ? overlap : 0));
    const int n = overlap + 1;
    for (int i = 1; i < n; ++i) r[i - 1] = (float)((double)i / n);  // img2img_load.cpp:35-38
    return r;
}

// ------------------------------------------------------------------------------------------------
// Antialiased bicubic weights: the kernel is stretched by s = max(n_in / n_out, 1), so a reduction by r reads about 4r + 1 inputs.
// ------------------------------------------------------------------------------------------------
ResampleAxis resampleAxis(int nIn, int nOut) {
    if (nIn < 1 || nOut < 1 || nOut > nIn) throw Error("resample: need 1 <= output size <= input size");
    auto cubic = [](double x) {
        const double a = -0.5;
        x = std::fabs(x);
        if (x < 1) return ((a + 2) * x - (a + 3)) * x * x + 1;
        if (x < 2) return a * (((x - 5) * x + 8) * x - 4);
        return 0.0;
    };
    const double r = (double)nIn / nOut, s = std::max(r, 1.0);
    ResampleAxis ax;
    ax.nIn = nIn;
    ax.nOut = nOut;
    ax.first.resize(nOut);
    ax.count.resize(nOut);
    std::vector<std::vector<double>> rows(nOut);
    for (int i = 0; i < nOut; ++i) {
        const double c = r * (i + 0.5);
        const int lo = std::max((int)std::floor(c - 2 * s + 0.5), 0), hi = std::min((int)std::floor(c + 2 * s + 0.5), nIn);
        std::vector<double>& wr = rows[i];
        double sum = 0;
        for (int j = lo; j < hi; ++j) {
            wr.push_back(cubic((j - c + 0.5) / s));
            sum += wr.back();
        }
        for (double& v : wr) v /= sum;
        int b = 0, e = (int)wr.size();
        while (e - b > 1 && wr[b] == 0.0) ++b;
        while (e - b > 1 && wr[e - 1] == 0.0) --e;
        wr = std::vector<double>(wr.begin() + b, wr.begin() + e);
        ax.first[i] = lo + b;
        ax.count[i] = e - b;
        ax.taps = std::max(ax.taps, e - b);
    }
    ax.w.assign((size_t)nOut * ax.taps, 0.f);
    for (int i = 0; i < nOut; ++i)
        for (int k = 0; k < ax.count[i]; ++k) ax.w[(size_t)i * ax.taps + k] = (float)rows[i][k];
    return ax;
}

// ------------------------------------------------------------------------------------------------
// SHA-256 (FIPS 180-4), written from the standard.
// ------------------------------------------------------------------------------------------------
namespace {
inline uint32_t rotr(uint32_t x, int n) { return (x >> n) | (x << (32 - n)); }
const uint32_t K256[64] = {
    0x428a2f98, 0x71374491, 0xb5c0fbcf, 0xe9b5dba5, 0x3956c25b, 0x59f111f1, 0x923f82a4, 0xab1c5ed5, 0xd807aa98,
    0x12835b01, 0x243185be, 0x550c7dc3, 0x72be5d74, 0x80deb1fe, 0x9bdc06a7, 0xc19bf174, 0xe49b69c1, 0xefbe4786,
    0x0fc19dc6, 0x240ca1cc, 0x2de92c6f, 0x4a7484aa, 0x5cb0a9dc, 0x76f988da, 0x983e5152, 0xa831c66d, 0xb00327c8,
    0xbf597fc7, 0xc6e00bf3, 0xd5a79147, 0x06ca6351, 0x14292967, 0x27b70a85, 0x2e1b2138, 0x4d2c6dfc, 0x53380d13,
    0x650a7354, 0x766a0abb, 0x81c2c92e, 0x92722c85, 0xa2bfe8a1, 0xa81a664b, 0xc24b8b70, 0xc76c51a3, 0xd192e819,
    0xd6990624, 0xf40e3585, 0x106aa070, 0x19a4c116, 0x1e376c08, 0x2748774c, 0x34b0bcb5, 0x391c0cb3, 0x4ed8aa4a,
    0x5b9cca4f, 0x682e6ff3, 0x748f82ee, 0x78a5636f, 0x84c87814, 0x8cc70208, 0x90befffa, 0xa4506ceb, 0xbef9a3f7,
    0xc67178f2};
}  // namespace

std::string sha256Hex(const std::string& data) {
    uint32_t h[8] = {0x6a09e667, 0xbb67ae85, 0x3c6ef372, 0xa54ff53a, 0x510e527f, 0x9b05688c, 0x1f83d9ab, 0x5be0cd19};
    std::vector<uint8_t> msg(data.begin(), data.end());
    const uint64_t bits = (uint64_t)msg.size() * 8;
    msg.push_back(0x80);
    while (msg.size() % 64 != 56) msg.push_back(0);
    for (int i = 7; i >= 0; --i) msg.push_back((uint8_t)(bits >> (8 * i)));
    for (size_t off = 0; off < msg.size(); off += 64) {
        uint32_t w[64];
        for (int t = 0; t < 16; ++t)
            w[t] = (uint32_t)msg[off + 4 * t] << 24 | (uint32_t)msg[off + 4 * t + 1] << 16 |
                   (uint32_t)msg[off + 4 * t + 2] << 8 | (uint32_t)msg[off + 4 * t + 3];
        for (int t = 16; t < 64; ++t) {
            const uint32_t s0 = rotr(w[t - 15], 7) ^ rotr(w[t - 15], 18) ^ (w[t - 15] >> 3);
            const uint32_t s1 = rotr(w[t - 2], 17) ^ rotr(w[t - 2], 19) ^ (w[t - 2] >> 10);
            w[t] = w[t - 16] + s0 + w[t - 7] + s1;
        }
        uint32_t a = h[0], b = h[1], c = h[2], d = h[3], e = h[4], f = h[5], g = h[6], hh = h[7];
        for (int t = 0; t < 64; ++t) {
            const uint32_t S1 = rotr(e, 6) ^ rotr(e, 11) ^ rotr(e, 25);
            const uint32_t ch = (e & f) ^ (~e & g);
            const uint32_t t1 = hh + S1 + ch + K256[t] + w[t];
            const uint32_t S0 = rotr(a, 2) ^ rotr(a, 13) ^ rotr(a, 22);
            const uint32_t mj = (a & b) ^ (a & c) ^ (b & c);
            const uint32_t t2 = S0 + mj;
            hh = g; g = f; f = e; e = d + t1; d = c; c = b; b = a; a = t1 + t2;
        }
        h[0] += a; h[1] += b; h[2] += c; h[3] += d; h[4] += e; h[5] += f; h[6] += g; h[7] += hh;
    }
    char out[65];
    for (int i = 0; i < 8; ++i) std::snprintf(out + 8 * i, 9, "%08x", h[i]);
    return std::string(out, 64);
}

// "<DeviceNameNoSpaces>.<FP16|TF32>.minB.optB.maxB.minC.optC.maxC.minW.optW.maxW.minH.optH.maxH"
// (img2img_build.cpp:8-27)
std::string configHashString(const std::string& deviceName, const w2x_build_config& c) {
    std::string dn;
    for (char ch : deviceName)
        if (!std::isspace((unsigned char)ch)) dn.push_back(ch);
    std::ostringstream o;
    o << dn << "." << (c.precision == W2X_PRECISION_FP16 ? "FP16" : "TF32") << ".";
    o << c.minBatchSize << "." << c.optBatchSize << "." << c.maxBatchSize << "." << c.minChannels << "."
      << c.optChannels << "." << c.maxChannels << "." << c.minWidth << "." << c.optWidth << "." << c.maxWidth << "."
      << c.minHeight << "." << c.optHeight << "." << c.maxHeight;
    return o.str();
}

std::string configHash(const std::string& deviceName, const w2x_build_config& c) {
    return sha256Hex(configHashString(deviceName, c));
}

// ------------------------------------------------------------------------------------------------
// JSON sidecar: a flat object of one string key ("deviceName"), one string enum ("precision") and
// twelve ints, written with 4-space indentation in the reference's key order (img2img_build.cpp:29-50).
// The reader accepts any flat JSON object of strings / integers in any order.
// ------------------------------------------------------------------------------------------------
static std::string jsonEscape(const std::string& s) {
    std::string o;
    for (char ch : s) {
        if (ch == '"' || ch == '\\') { o.push_back('\\'); o.push_back(ch); }
        else if (ch == '\n') o += "\\n";
        else o.push_back(ch);
    }
    return o;
}

void writeSidecar(const std::string& path, const Sidecar& s) {
    std::ofstream f(path);
    if (!f.is_open()) throw Error("could not open config \"" + path + "\"");
    const w2x_build_config& c = s.cfg;
    f << "{\n";
    f << "    \"deviceName\": \"" << jsonEscape(s.deviceName) << "\",\n";
    f << "    \"precision\": \"" << (c.precision == W2X_PRECISION_FP16 ? "FP16" : "TF32") << "\",\n";
    const std::pair<const char*, int> kv[] = {
        {"minBatchSize", c.minBatchSize}, {"optBatchSize", c.optBatchSize}, {"maxBatchSize", c.maxBatchSize},
        {"minChannels", c.minChannels},   {"optChannels", c.optChannels},   {"maxChannels", c.maxChannels},
        {"minWidth", c.minWidth},         {"optWidth", c.optWidth},         {"maxWidth", c.maxWidth},
        {"minHeight", c.minHeight},       {"optHeight", c.optHeight},       {"maxHeight", c.maxHeight}};
    for (size_t i = 0; i < 12; ++i)
        f << "    \"" << kv[i].first << "\": " << kv[i].second << (i + 1 < 12 ? ",\n" : "\n");
    f << "}";
}

namespace {
struct JsonFlat {
    std::map<std::string, std::string> str;
    std::map<std::string, long long> num;
};

JsonFlat parseFlatJson(const std::string& t) {
    JsonFlat out;
    size_t i = 0;
    auto ws = [&] { while (i < t.size() && std::isspace((unsigned char)t[i])) ++i; };
    auto str = [&]() -> std::string {
        if (t[i] != '"') throw Error("json: expected string");
        ++i;
        std::string s;
        while (i < t.size() && t[i] != '"') {
            if (t[i] == '\\' && i + 1 < t.size()) {
                ++i;
                s.push_back(t[i] == 'n' ? '\n' : t[i]);
            } else s.push_back(t[i]);
            ++i;
        }
        if (i >= t.size()) throw Error("json: unterminated string");
        ++i;
        return s;
    };
    ws();
    if (i >= t.size() || t[i] != '{') throw Error("json: expected object");
    ++i;
    for (;;) {
        ws();
        if (i < t.size() && t[i] == '}') break;
        std::string key = str();
        ws();
        if (i >= t.size() || t[i] != ':') throw Error("json: expected ':'");
        ++i;
        ws();
        if (i < t.size() && t[i] == '"') out.str[key] = str();
        else {
            size_t j = i;
            while (j < t.size() && (std::isdigit((unsigned char)t[j]) || t[j] == '-' || t[j] == '+')) ++j;
            if (j == i) throw Error("json: unsupported value for key " + key);
            out.num[key] = std::stoll(t.substr(i, j - i));
            i = j;
        }
        ws();
        if (i < t.size() && t[i] == ',') { ++i; continue; }
        ws();
        if (i < t.size() && t[i] == '}') break;
        throw Error("json: expected ',' or '}'");
    }
    return out;
}
}  // namespace

Sidecar readSidecar(const std::string& path) {
    std::ifstream f(path);
    if (!f.is_open()) throw Error("could not open config \"" + path + "\"");
    std::stringstream ss;
    ss << f.rdbuf();
    JsonFlat j = parseFlatJson(ss.str());
    auto S = [&](const char* k) -> std::string {
        auto it = j.str.find(k);
        if (it == j.str.end()) throw Error(std::string("json: missing key ") + k);
        return it->second;
    };
    auto N = [&](const char* k) -> int {
        auto it = j.num.find(k);
        if (it == j.num.end()) throw Error(std::string("json: missing key ") + k);
        return (int)it->second;
    };
    Sidecar s;
    s.deviceName = S("deviceName");
    s.cfg.deviceId = -1;  // resolved by the caller via device-name lookup (img2img_load.cpp:62-63)
    s.cfg.precision = S("precision") == "FP16" ? W2X_PRECISION_FP16 : W2X_PRECISION_TF32;
    s.cfg.minBatchSize = N("minBatchSize"); s.cfg.optBatchSize = N("optBatchSize"); s.cfg.maxBatchSize = N("maxBatchSize");
    s.cfg.minChannels = N("minChannels");   s.cfg.optChannels = N("optChannels");   s.cfg.maxChannels = N("maxChannels");
    s.cfg.minWidth = N("minWidth");         s.cfg.optWidth = N("optWidth");         s.cfg.maxWidth = N("maxWidth");
    s.cfg.minHeight = N("minHeight");       s.cfg.optHeight = N("optHeight");       s.cfg.maxHeight = N("maxHeight");
    return s;
}

bool isCompatible(const w2x_render_config& r, const w2x_build_config& b) {
    return r.deviceId == b.deviceId && r.precision == b.precision && r.batchSize >= b.minBatchSize &&
           r.batchSize <= b.maxBatchSize && r.channels >= b.minChannels && r.channels <= b.maxChannels &&
           r.width >= b.minWidth && r.width <= b.maxWidth && r.height >= b.minHeight && r.height <= b.maxHeight;
}

bool isOptimized(const w2x_render_config& r, const w2x_build_config& b) {
    return r.batchSize == b.optBatchSize && r.channels == b.optChannels && r.width == b.optWidth &&
           r.height == b.optHeight;
}

// getEnginePath, img2img_load.cpp:79-114: among the artefacts "<stem>_<16 hex>.w2x" next to the model that have a json sidecar
// and are compatible with the render configuration, an optimized one (opt == requested) wins, else the first compatible one.
// Deviations (SURVEY q6 and 8e): the file name must match exactly (the reference's prefix match lets "noise0" pick up
// "noise0_scale2x_<hash>"), candidates are visited in sorted order so the choice is deterministic, and a plan is compatible
// with EVERY device that carries the recorded device name -- the reference maps the name back to the first such device
// (helper.h:47-56), so on a box of identical GPUs only device 0 could ever load an engine.
std::string selectEngine(const std::string& modelPath, const w2x_render_config& rc, const std::string& rcDeviceName) {
    namespace fs = std::filesystem;
    if (!fs::exists(modelPath)) throw Error("model file does not exist");
    const std::string stem = fs::path(modelPath).stem().string();
    fs::path dir = fs::path(modelPath).parent_path();
    if (dir.empty()) dir = ".";
    std::vector<fs::path> cands;
    for (const auto& entry : fs::directory_iterator(dir)) {
        if (!entry.is_regular_file()) continue;
        const fs::path& p = entry.path();
        const std::string fn = p.filename().string();
        if (p.extension().string() != ".w2x" || fn.size() != stem.size() + 1 + 16 + 4) continue;
        if (fn.compare(0, stem.size(), stem) != 0 || fn[stem.size()] != '_') continue;
        bool hex = true;
        for (size_t i = stem.size() + 1; i < stem.size() + 17; ++i) hex = hex && std::isxdigit((unsigned char)fn[i]);
        if (hex) cands.push_back(p);
    }
    std::sort(cands.begin(), cands.end());
    std::string chosen;
    for (const auto& p : cands) {
        const std::string cfgPath = fs::path(p).replace_extension("").string() + ".json";
        if (!fs::exists(cfgPath)) continue;
        Sidecar sc = readSidecar(cfgPath);
        sc.cfg.deviceId = (!rcDeviceName.empty() && sc.deviceName == rcDeviceName) ? rc.deviceId : -1;
        if (isCompatible(rc, sc.cfg)) {
            if (isOptimized(rc, sc.cfg)) return p.string();
            if (chosen.empty()) chosen = p.string();
        }
    }
    if (chosen.empty()) throw Error("could not satisfy render configuration");
    return chosen;
}

std::vector<uint8_t> readFile(const std::string& path) {
    std::ifstream f(path, std::ios::binary | std::ios::ate);
    if (!f.is_open()) throw Error("could not open file \"" + path + "\"");
    const std::streamsize n = f.tellg();
    std::vector<uint8_t> buf((size_t)n);
    f.seekg(0, std::ios::beg);
    f.read((char*)buf.data(), n);
    return buf;
}

void writeFile(const std::string& path, const void* data, size_t n) {
    std::ofstream f(path, std::ios::binary);
    if (!f.is_open()) throw Error("could not open file \"" + path + "\" for writing");
    f.write((const char*)data, (std::streamsize)n);
    if (!f.good()) throw Error("short write to \"" + path + "\"");
}

}  // namespace w2x
