// Host-side utilities: tile grid arithmetic, sha256, flat-JSON sidecar, file helpers.
// Restates (does not copy) the host logic of /root/reference/src/tensorrt/img2img_{render,load,build}.cpp.
#pragma once
#include <cstdint>
#include <map>
#include <cstdlib>
#include <stdexcept>
#include <string>
#include <vector>

#include "../../include/w2x.h"

namespace w2x {

struct Error : std::runtime_error {
    using std::runtime_error::runtime_error;
};

// Development switches (kernel variants, timing experiments that skip work) exist only in the W2X_DEV build (lib/libw2x_dev.so);
// the shipped library ignores the environment for them.
inline const char* devEnv(const char* name) {
#ifdef W2X_DEV
    return std::getenv(name);
#else
    (void)name;
    return nullptr;
#endif
}

// ---- tile grid (img2img_render.cpp:7-66) ----------------------------------------------------------
struct TileGrid {
    int count = 0, nx = 0, ny = 0;
    int scaledInW = 0, scaledInH = 0;     // scaledInputTileSize
    int inOvX = 0, inOvY = 0;             // inputOverlap
    int outOvX = 0, outOvY = 0;           // scaledOutputOverlap
    std::vector<w2x_rect> inRects, outRects;  // column-major: index = i * ny + j
};

TileGrid calculateTiles(int inW, int inH, int outW, int outH, int tileW, int tileH, int outTileW, int outTileH,
                        int scaling, double overlapX, double overlapY);

// createTileWeights (img2img_load.cpp:29-52): ramp[i] = float(double(i + 1) / double(overlap + 1)), i in [0, overlap)
std::vector<float> blendRamp(int overlap);

// ---- antialiased bicubic reduction (w2x_render_resized) --------------------------------------------
// One axis n_in -> n_out (1 <= n_out <= n_in): output index i reads inputs first[i] .. first[i] + count[i] - 1 with weights
// w[i * taps + k] (k < count[i]; the rest of the row is 0).  The weights are torch's interpolate(mode="bicubic", antialias=True,
// align_corners=False), i.e. PIL's BICUBIC (a = -0.5), computed in double, normalised to sum 1 and stored as float; zero weights at
// either end of a window are dropped, so an identity axis is one tap of weight 1.  first[i] and first[i] + count[i] never decrease.
struct ResampleAxis {
    int nIn = 0, nOut = 0, taps = 0;
    std::vector<int> first, count;
    std::vector<float> w;
};
ResampleAxis resampleAxis(int nIn, int nOut);   // throws Error outside 1 <= nOut <= nIn

// ---- sha256 (lowercase hex), json sidecar, naming (img2img_build.cpp:8-50,151-154; img2img_load.cpp:54-114) -----
std::string sha256Hex(const std::string& data);
std::string configHashString(const std::string& deviceName, const w2x_build_config& c);  // pre-hash string
std::string configHash(const std::string& deviceName, const w2x_build_config& c);        // sha256 hex

struct Sidecar {
    std::string deviceName;
    w2x_build_config cfg{};
};
void writeSidecar(const std::string& path, const Sidecar& s);
Sidecar readSidecar(const std::string& path);

bool isCompatible(const w2x_render_config& r, const w2x_build_config& b);  // img2img_load.cpp:9-20
bool isOptimized(const w2x_render_config& r, const w2x_build_config& b);
// engine artefact discovery (img2img_load.cpp:79-114) for a render on a device called rcDeviceName; throws when nothing fits
std::string selectEngine(const std::string& modelPath, const w2x_render_config& rc, const std::string& rcDeviceName);   // img2img_load.cpp:22-27

std::vector<uint8_t> readFile(const std::string& path);
void writeFile(const std::string& path, const void* data, size_t n);

}  // namespace w2x
