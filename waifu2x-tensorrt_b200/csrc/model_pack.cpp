#include "model_pack.h"

#include <cmath>
#include <algorithm>
#include <cstring>
#include <deque>

#include "hostutil.h"

namespace w2x {

// ------------------------------------------------------------------------------------------------
// fp16 <-> fp32 on the host (round-to-nearest-even), so packing needs no CUDA.
// ------------------------------------------------------------------------------------------------
uint16_t floatToHalfBits(float f) {
    uint32_t x;
    std::memcpy(&x, &f, 4);
    const uint32_t sign = (x >> 16) & 0x8000u;
    x &= 0x7fffffffu;
    if (x >= 0x7f800000u) return (uint16_t)(sign | 0x7c00u | (x > 0x7f800000u ? 0x200u : 0));  // inf / nan
    if (x >= 0x477ff000u) return (uint16_t)(sign | 0x7c00u);                                     // overflow -> inf
    if (x < 0x33000001u) return (uint16_t)sign;                                                  // underflow -> 0
    int e = (int)(x >> 23) - 127;
    uint32_t m = x & 0x7fffffu;
    if (e < -14) {  // subnormal half
        m |= 0x800000u;
        const int shift = -14 - e + 13;  // bits to drop
        const uint32_t rem = m & ((1u << shift) - 1), half = 1u << (shift - 1);
        uint32_t r = m >> shift;
        if (rem > half || (rem == half && (r & 1))) ++r;
        return (uint16_t)(sign | r);
    }
    uint32_t r = ((uint32_t)(e + 15) << 10) | (m >> 13);
    const uint32_t rem = m & 0x1fffu;
    if (rem > 0x1000u || (rem == 0x1000u && (r & 1))) ++r;  // carries into the exponent correctly
    return (uint16_t)(sign | r);
}

float halfBitsToFloat(uint16_t h) {
    const uint32_t sign = (uint32_t)(h & 0x8000u) << 16;
    uint32_t e = (h >> 10) & 0x1f, m = h & 0x3ffu, x;
    if (e == 0) {
        if (m == 0) x = sign;
        else {
            int s = 0;
            while (!(m & 0x400u)) { m <<= 1; ++s; }
            m &= 0x3ffu;
            x = sign | ((uint32_t)(127 - 15 - s + 1) << 23) | (m << 13);
        }
    } else if (e == 31) x = sign | 0x7f800000u | (m << 13);
    else x = sign | ((e + 112) << 23) | (m << 13);
    float f;
    std::memcpy(&f, &x, 4);
    return f;
}

// ------------------------------------------------------------------------------------------------
// Protobuf wire-format reader (just enough for ONNX ModelProto / GraphProto / NodeProto / TensorProto).
// ------------------------------------------------------------------------------------------------
namespace {
struct Span {
    const uint8_t* p;
    size_t n;
};
struct Field {
    uint32_t id, wt;
    uint64_t v;   // varint / fixed
    Span bytes;   // length-delimited
};
struct Reader {
    const uint8_t* p;
    const uint8_t* end;
    explicit Reader(Span s) : p(s.p), end(s.p + s.n) {}
    bool done() const { return p >= end; }
    uint64_t varint() {
        uint64_t v = 0;
        int s = 0;
        while (true) {
            if (p >= end) throw Error("onnx: truncated varint");
            const uint8_t c = *p++;
            v |= (uint64_t)(c & 0x7f) << s;
            if (!(c & 0x80)) return v;
            s += 7;
            if (s > 63) throw Error("onnx: varint too long");
        }
    }
    Field next() {
        Field f{};
        const uint64_t key = varint();
        f.id = (uint32_t)(key >> 3);
        f.wt = (uint32_t)(key & 7);
        switch (f.wt) {
            case 0: f.v = varint(); break;
            case 1:
                if (end - p < 8) throw Error("onnx: truncated fixed64");
                std::memcpy(&f.v, p, 8); p += 8; break;
            case 5: {
                if (end - p < 4) throw Error("onnx: truncated fixed32");
                uint32_t t; std::memcpy(&t, p, 4); f.v = t; p += 4; break;
            }
            case 2: {
                const uint64_t n = varint();
                if ((uint64_t)(end - p) < n) throw Error("onnx: truncated bytes field");
                f.bytes = {p, (size_t)n};
                p += n;
                break;
            }
            default: throw Error("onnx: unsupported wire type");
        }
        return f;
    }
};

std::string str(Span s) { return std::string((const char*)s.p, s.n); }

void readInts(const Field& f, std::vector<int64_t>& out) {
    if (f.wt == 2) {
        Reader r(f.bytes);
        while (!r.done()) out.push_back((int64_t)r.varint());
    } else out.push_back((int64_t)f.v);
}

OnnxTensor parseTensor(Span s) {
    OnnxTensor t;
    int dtype = 1;
    Span raw{nullptr, 0};
    std::vector<float> fdata;
    std::vector<double> ddata;
    Reader r(s);
    while (!r.done()) {
        Field f = r.next();
        switch (f.id) {
            case 1: readInts(f, t.dims); break;
            case 2: dtype = (int)f.v; break;
            case 4:
                if (f.wt == 2) {
                    for (size_t i = 0; i + 4 <= f.bytes.n; i += 4) { float v; std::memcpy(&v, f.bytes.p + i, 4); fdata.push_back(v); }
                } else { uint32_t u = (uint32_t)f.v; float v; std::memcpy(&v, &u, 4); fdata.push_back(v); }
                break;
            case 7: readInts(f, t.idata); break;
            case 8: t.name = str(f.bytes); break;
            case 9: raw = f.bytes; break;
            case 10:
                if (f.wt == 2) {
                    for (size_t i = 0; i + 8 <= f.bytes.n; i += 8) { double v; std::memcpy(&v, f.bytes.p + i, 8); ddata.push_back(v); }
                } else { double v; std::memcpy(&v, &f.v, 8); ddata.push_back(v); }
                break;
            default: break;
        }
    }
    if (dtype == 1) {  // FLOAT
        if (raw.n) { t.data.resize(raw.n / 4); std::memcpy(t.data.data(), raw.p, t.data.size() * 4); }
        else t.data = fdata;
    } else if (dtype == 10) {  // FLOAT16
        t.data.resize(raw.n / 2);
        for (size_t i = 0; i < t.data.size(); ++i) { uint16_t h; std::memcpy(&h, raw.p + 2 * i, 2); t.data[i] = halfBitsToFloat(h); }
    } else if (dtype == 11) {  // DOUBLE
        if (raw.n) { t.data.resize(raw.n / 8); for (size_t i = 0; i < t.data.size(); ++i) { double d; std::memcpy(&d, raw.p + 8 * i, 8); t.data[i] = (float)d; } }
        else for (double d : ddata) t.data.push_back((float)d);
    } else if (dtype == 7) {  // INT64
        if (raw.n) { t.idata.resize(raw.n / 8); std::memcpy(t.idata.data(), raw.p, t.idata.size() * 8); }
    }
    return t;
}

OnnxNode parseNode(Span s, std::vector<OnnxTensor>& constants) {
    OnnxNode n;
    std::vector<Span> attrs;
    Reader r(s);
    while (!r.done()) {
        Field f = r.next();
        switch (f.id) {
            case 1: n.inputs.push_back(str(f.bytes)); break;
            case 2: n.outputs.push_back(str(f.bytes)); break;
            case 3: n.name = str(f.bytes); break;
            case 4: n.op = str(f.bytes); break;
            case 5: attrs.push_back(f.bytes); break;
            default: break;
        }
    }
    for (Span a : attrs) {
        std::string an, sval;
        std::vector<int64_t> ints;
        Span tens{nullptr, 0};
        float fval = 0.f;
        int64_t ival = 0;
        Reader ar(a);
        while (!ar.done()) {
            Field f = ar.next();
            if (f.id == 1) an = str(f.bytes);
            else if (f.id == 2 && f.wt == 5) { uint32_t u = (uint32_t)f.v; std::memcpy(&fval, &u, 4); }
            else if (f.id == 3 && f.wt == 0) ival = (int64_t)f.v;
            else if (f.id == 4 && f.wt == 2) sval = str(f.bytes);
            else if (f.id == 8) readInts(f, ints);
            else if (f.id == 5 && f.wt == 2) tens = f.bytes;
        }
        if (an == "kernel_shape") n.kernel_shape = ints;
        else if (an == "strides") n.strides = ints;
        else if (an == "pads") n.pads = ints;
        else if (an == "dilations") n.dilations = ints;
        else if (an == "axes") n.axes = ints;
        else if (an == "group") n.group = ival;
        else if (an == "transA") n.transA = ival;
        else if (an == "transB") n.transB = ival;
        else if (an == "auto_pad") n.auto_pad = sval;
        else if (an == "alpha") n.alpha = fval;
        else if (an == "min") { n.hasMin = true; n.minv = fval; }
        else if (an == "max") { n.hasMax = true; n.maxv = fval; }
        else if (an == "epsilon") n.epsilon = fval;
        else if (an == "value" && n.op == "Constant" && tens.p && !n.outputs.empty()) {
            OnnxTensor t = parseTensor(tens);
            t.name = n.outputs[0];
            constants.push_back(std::move(t));
        }
    }
    return n;
}
}  // namespace

const OnnxTensor* OnnxGraph::find(const std::string& name) const {
    for (const auto& t : initializers)
        if (t.name == name) return &t;
    return nullptr;
}

OnnxGraph parseOnnx(const std::vector<uint8_t>& blob) {
    Span graph{nullptr, 0};
    {
        Reader r(Span{blob.data(), blob.size()});
        while (!r.done()) {
            Field f = r.next();
            if (f.id == 7 && f.wt == 2) graph = f.bytes;
        }
    }
    if (!graph.p) throw Error("onnx: no graph in model");
    OnnxGraph g;
    Reader r(graph);
    while (!r.done()) {
        Field f = r.next();
        if (f.id == 1 && f.wt == 2) g.nodes.push_back(parseNode(f.bytes, g.initializers));
        else if (f.id == 5 && f.wt == 2) g.initializers.push_back(parseTensor(f.bytes));
    }
    return g;
}

// ------------------------------------------------------------------------------------------------
// Architecture template match + packing.
// ------------------------------------------------------------------------------------------------
namespace {
struct ConvNode {
    std::string name;
    bool transpose = false;
    int cout = 0, cin = 0, kh = 0, kw = 0, stride = 1, pad = 0;
    const OnnxTensor* w = nullptr;
    const OnnxTensor* b = nullptr;
    const OnnxNode* node = nullptr;
};

// ---- topology checks: the kernels hard-wire what the weight shapes cannot tell (activation slope, crops, clamp) ---------------
struct GraphIndex {
    const OnnxGraph& g;
    explicit GraphIndex(const OnnxGraph& g_) : g(g_) {}
    // nodes that read tensor `name`, looking through Identity / Cast
    std::vector<const OnnxNode*> consumers(const std::string& name) const {
        std::vector<const OnnxNode*> out;
        for (const auto& n : g.nodes)
            for (const auto& in : n.inputs)
                if (in == name) {
                    if ((n.op == "Identity" || n.op == "Cast") && !n.outputs.empty()) {
                        auto more = consumers(n.outputs[0]);
                        out.insert(out.end(), more.begin(), more.end());
                    } else {
                        out.push_back(&n);
                    }
                }
        return out;
    }
    const OnnxNode* producer(const std::string& name) const {
        for (const auto& n : g.nodes)
            for (const auto& o : n.outputs)
                if (o == name) return &n;
        return nullptr;
    }
    const OnnxNode* consumerOp(const std::string& name, const char* op) const {
        for (const OnnxNode* n : consumers(name))
            if (n->op == op) return n;
        return nullptr;
    }
};

// symmetric spatial crop amount of a Slice (starts [p,p], ends [-p,-p] over axes 2,3) or a negative Pad; -1 if the node is neither
int cropAmount(const OnnxGraph& g, const OnnxNode& n) {
    if (n.op == "Slice" && n.inputs.size() >= 3) {
        const OnnxTensor *s = g.find(n.inputs[1]), *e = g.find(n.inputs[2]);
        const OnnxTensor* ax = n.inputs.size() > 3 ? g.find(n.inputs[3]) : nullptr;
        if (!s || !e || s->idata.size() != 2 || e->idata.size() != 2) return -1;
        if (ax && (ax->idata.size() != 2 || !((ax->idata[0] == 2 && ax->idata[1] == 3) || (ax->idata[0] == -2 && ax->idata[1] == -1)))) return -1;
        if (s->idata[0] != s->idata[1] || e->idata[0] != e->idata[1] || s->idata[0] <= 0 || e->idata[0] != -s->idata[0]) return -1;
        return (int)s->idata[0];
    }
    if (n.op == "Pad") {
        std::vector<int64_t> pads = n.pads;
        if (pads.empty() && n.inputs.size() >= 2)
            if (const OnnxTensor* p = g.find(n.inputs[1])) pads = p->idata;
        if (pads.size() != 8 || pads[0] || pads[1] || pads[4] || pads[5]) return -1;
        if (pads[2] >= 0 || pads[2] != pads[3] || pads[2] != pads[6] || pads[2] != pads[7]) return -1;
        return (int)-pads[2];
    }
    return -1;
}

void verifyClip01(const OnnxGraph& g, const char* what) {
    for (const auto& n : g.nodes) {
        if (n.op != "Clip") continue;
        float lo = n.minv, hi = n.maxv;
        bool haveLo = n.hasMin, haveHi = n.hasMax;
        if (n.inputs.size() > 1 && !n.inputs[1].empty())
            if (const OnnxTensor* t = g.find(n.inputs[1])) { if (!t->data.empty()) { lo = t->data[0]; haveLo = true; } }
        if (n.inputs.size() > 2 && !n.inputs[2].empty())
            if (const OnnxTensor* t = g.find(n.inputs[2])) { if (!t->data.empty()) { hi = t->data[0]; haveHi = true; } }
        if (haveLo && haveHi && lo == 0.f && hi == 1.f) return;
        throw Error(std::string("pack: ") + what + " clamps its output to something other than [0, 1]");
    }
    throw Error(std::string("pack: ") + what + " has no Clip(0, 1) on its output (the image head kernels clamp unconditionally)");
}

std::vector<ConvNode> collectConvs(const OnnxGraph& g) {
    std::vector<ConvNode> out;
    for (const auto& n : g.nodes) {
        if (n.op != "Conv" && n.op != "ConvTranspose") continue;
        if (n.inputs.size() < 2) throw Error("onnx: conv node without weight input");
        ConvNode c;
        c.name = n.name;
        c.transpose = n.op == "ConvTranspose";
        c.w = g.find(n.inputs[1]);
        if (!c.w || c.w->dims.size() != 4) throw Error("onnx: conv weight '" + n.inputs[1] + "' is not a 4-d initializer");
        if (n.inputs.size() > 2 && !n.inputs[2].empty()) c.b = g.find(n.inputs[2]);
        const auto& d = c.w->dims;
        c.cout = (int)(c.transpose ? d[1] : d[0]);
        c.cin = (int)(c.transpose ? d[0] : d[1]);
        c.kh = (int)d[2];
        c.kw = (int)d[3];
        c.stride = n.strides.empty() ? 1 : (int)n.strides[0];
        c.pad = n.pads.empty() ? 0 : (int)n.pads[0];
        // the kernels implement plain dense convolutions only: anything else must fail the build, not run wrong
        if (n.group != 1) throw Error("onnx: conv '" + n.name + "' has group " + std::to_string(n.group) + " (only 1 is supported)");
        for (int64_t d : n.dilations)
            if (d != 1) throw Error("onnx: conv '" + n.name + "' is dilated (unsupported)");
        for (int64_t s : n.strides)
            if (s != c.stride) throw Error("onnx: conv '" + n.name + "' has anisotropic strides (unsupported)");
        for (int64_t p : n.pads)
            if (p != c.pad) throw Error("onnx: conv '" + n.name + "' has asymmetric padding (unsupported)");
        if (!n.auto_pad.empty() && n.auto_pad != "NOTSET") throw Error("onnx: conv '" + n.name + "' uses auto_pad " + n.auto_pad + " (unsupported)");
        c.node = &n;
        if ((size_t)(d[0] * d[1] * d[2] * d[3]) != c.w->data.size()) throw Error("onnx: conv weight '" + c.w->name + "' has no float data");
        out.push_back(c);
    }
    return out;
}

inline float W4(const OnnxTensor* t, int a, int b, int c, int d) {
    const auto& s = t->dims;
    return t->data[(((size_t)a * s[1] + b) * s[2] + c) * s[3] + d];
}

// tf32: the GEMM weights are stored as fp32 rounded to nearest TF32 (PackedLayer::wf) instead of fp16 bits (PackedLayer::w)
PackedLayer packLayer(const ConvNode& c, bool tf32, int cinStore = 0, int npadTo = 0) {
    PackedLayer L;
    L.name = c.name;
    L.cout = (uint32_t)c.cout;
    const int cinp = cinStore > 0 ? cinStore : (c.cin < 8 ? 4 : c.cin);  // RGB first layers are stored with 4 channels
    if (cinp < c.cin || (cinp % 4)) throw Error("pack: unsupported cin in " + c.name);
    L.cin = (uint32_t)cinp;
    auto bias = [&](int co) { return c.b ? c.b->data[(size_t)co] : 0.0f; };
    std::vector<float> w;  // [npad][ktot]
    if (!c.transpose && c.kh == 3 && c.kw == 3 && c.stride == 1 && c.pad == 0) {
        L.kind = L_CONV3; L.taps = 9;
        L.npad = (uint32_t)(npadTo > 0 ? npadTo : (c.cout + 15) / 16 * 16);
        L.ktot = 9 * L.cin;
        w.assign((size_t)L.npad * L.ktot, 0.f);
        L.bias.assign(L.npad, 0.f);
        for (int co = 0; co < c.cout; ++co) {
            L.bias[co] = bias(co);
            for (int ky = 0; ky < 3; ++ky)
                for (int kx = 0; kx < 3; ++kx)
                    for (int ci = 0; ci < c.cin; ++ci)
                        w[(size_t)co * L.ktot + (ky * 3 + kx) * L.cin + ci] = W4(c.w, co, ci, ky, kx);
        }
    } else if (!c.transpose && c.kh == 2 && c.kw == 2 && c.stride == 2 && c.pad == 0) {
        L.kind = L_DOWN2; L.taps = 4;
        L.npad = (uint32_t)((c.cout + 15) / 16 * 16);
        L.ktot = 4 * L.cin;
        w.assign((size_t)L.npad * L.ktot, 0.f);
        L.bias.assign(L.npad, 0.f);
        for (int co = 0; co < c.cout; ++co) {
            L.bias[co] = bias(co);
            for (int dy = 0; dy < 2; ++dy)
                for (int dx = 0; dx < 2; ++dx)
                    for (int ci = 0; ci < c.cin; ++ci)
                        w[(size_t)co * L.ktot + (dy * 2 + dx) * L.cin + ci] = W4(c.w, co, ci, dy, dx);
        }
    } else if (c.transpose && c.kh == 2 && c.kw == 2 && c.stride == 2 && c.pad == 0) {
        if (c.cout % 8) throw Error("pack: convT 2x2 cout must be a multiple of 8 in " + c.name);
        L.kind = L_UP2; L.taps = 1;
        L.npad = (uint32_t)(4 * c.cout);
        L.ktot = L.cin;
        w.assign((size_t)L.npad * L.ktot, 0.f);
        L.bias.assign(L.npad, 0.f);
        for (int q = 0; q < 4; ++q)
            for (int co = 0; co < c.cout; ++co) {
                const int n = q * c.cout + co;
                L.bias[n] = bias(co);
                for (int ci = 0; ci < c.cin; ++ci)
                    w[(size_t)n * L.ktot + ci] = W4(c.w, ci, co, q >> 1, q & 1);
            }
    } else if (c.transpose && c.kh == 4 && c.kw == 4 && c.stride == 2 && c.pad == 3) {
        if (c.cout > 4) throw Error("pack: convT 4x4 head supports cout <= 4 in " + c.name);
        L.kind = L_UP4; L.taps = 4;
        L.npad = 16;
        L.ktot = 4 * L.cin;
        w.assign((size_t)L.npad * L.ktot, 0.f);
        L.bias.assign(L.npad, 0.f);
        for (int py = 0; py < 2; ++py)
            for (int px = 0; px < 2; ++px)
                for (int co = 0; co < c.cout; ++co) {
                    const int n = (py * 2 + px) * 4 + co;
                    L.bias[n] = bias(co);
                    for (int wy = 0; wy < 2; ++wy)
                        for (int wx = 0; wx < 2; ++wx)
                            for (int ci = 0; ci < c.cin; ++ci)
                                w[(size_t)n * L.ktot + (wy * 2 + wx) * L.cin + ci] =
                                    W4(c.w, ci, co, 2 + py - 2 * wy, 2 + px - 2 * wx);
                }
    } else {
        throw Error("pack: unsupported convolution '" + c.name + "' (k=" + std::to_string(c.kh) + " s=" +
                    std::to_string(c.stride) + " p=" + std::to_string(c.pad) + (c.transpose ? " transposed)" : ")"));
    }
    if (tf32) {
        L.wf.resize(w.size());
        for (size_t i = 0; i < w.size(); ++i) L.wf[i] = roundToTf32(w[i]);
    } else {
        L.w.resize(w.size());
        for (size_t i = 0; i < w.size(); ++i) L.w[i] = floatToHalfBits(w[i]);
    }
    return L;
}

struct Expect { uint32_t kind; int cin, cout; bool se; };

// ---- SwinUNet: weight-bearing nodes in graph order -> typed records ------------------------------------------------
PackedLayer packLinear(const std::string& name, const OnnxTensor* w, const OnnxTensor* b, uint32_t kind, int cout4 = 0, int upscale = 0) {
    // ONNX MatMul weight is [K, N] (torch weight transposed)
    if (!w || w->dims.size() != 2) throw Error("pack: MatMul weight of '" + name + "' is not a 2-d initializer");
    const int K = (int)w->dims[0], N = (int)w->dims[1];
    if ((size_t)K * N != w->data.size()) throw Error("pack: MatMul weight of '" + name + "' has no float data");
    if (K % 32) throw Error("pack: linear '" + name + "' needs K % 32 == 0");
    PackedLayer L;
    L.name = name;
    L.kind = kind;
    L.cin = (uint32_t)K; L.ktot = (uint32_t)K; L.taps = 1;
    auto W = [&](int k, int n) { return w->data[(size_t)k * N + n]; };
    auto B = [&](int n) { return b ? b->data[(size_t)n] : 0.f; };
    if (kind == L_LINEAR) {
        if (N % 16) throw Error("pack: linear '" + name + "' needs N % 16 == 0");
        L.cout = (uint32_t)N; L.npad = (uint32_t)N;
        L.w.assign((size_t)N * K, 0); L.bias.assign(N, 0.f);
        for (int n = 0; n < N; ++n) {
            L.bias[n] = B(n);
            for (int k = 0; k < K; ++k) L.w[(size_t)n * K + k] = floatToHalfBits(W(k, n));
        }
    } else if (kind == L_UPLIN) {  // pixel_shuffle(2): torch channel index c*4 + i*2 + j  ->  row (i*2+j)*cout + c
        if (N % 4 || (N / 4) % 8) throw Error("pack: PatchUp '" + name + "' has an unsupported width");
        const int cout = N / 4;
        L.cout = (uint32_t)cout; L.npad = (uint32_t)N;
        L.w.assign((size_t)N * K, 0); L.bias.assign(N, 0.f);
        for (int q = 0; q < 4; ++q)
            for (int c = 0; c < cout; ++c) {
                const int src = c * 4 + q, dst = q * cout + c;
                L.bias[dst] = B(src);
                for (int k = 0; k < K; ++k) L.w[(size_t)dst * K + k] = floatToHalfBits(W(k, src));
            }
    } else {  // L_TOIMG: N = 3*s*s -> 16 rows, row (i*2+j)*4 + c  (s = 1: row c)
        const int s = upscale;
        if (N != 3 * s * s || (s != 1 && s != 2)) throw Error("pack: ToImage '" + name + "' has an unsupported width");
        L.cout = 3; L.npad = 16; L.upscale = (uint32_t)s;
        L.w.assign((size_t)16 * K, 0); L.bias.assign(16, 0.f);
        for (int c = 0; c < 3; ++c)
            for (int q = 0; q < s * s; ++q) {
                const int src = c * s * s + q, dst = q * 4 + c;
                L.bias[dst] = B(src);
                for (int k = 0; k < K; ++k) L.w[(size_t)dst * K + k] = floatToHalfBits(W(k, src));
            }
    }
    (void)cout4;
    return L;
}

PackedModel packSwin(const OnnxGraph& g, int precision) {
    PackedModel m;
    m.precision = (uint32_t)precision;
    m.arch = ARCH_SWINUNET;
    // pass 1: collect records in node order
    struct Rec { int type; ConvNode conv; const OnnxTensor *a = nullptr, *b = nullptr; std::string name; float eps = 1e-5f; };
    enum { R_CONV, R_LN, R_LIN, R_ATTN };
    std::vector<Rec> recs;
    std::vector<ConvNode> convs = collectConvs(g);
    size_t ci = 0;
    int pendingLin = -1;
    std::string pendingOut;
    const GraphIndex gi(g);
    std::deque<OnnxTensor> synth;  // Gemm weights stored [N, K] (transB = 1), transposed into the MatMul convention
    // decomposed LayerNorm (exporters below opset 17): ... -> Div(x - mean, Sqrt(var + eps)) -> Mul(gamma) -> Add(beta)
    struct PendingLn { std::string mulOut; const OnnxTensor* gamma; float eps; };
    std::vector<PendingLn> pendingLn;
    auto isVec = [](const OnnxTensor* t) { return t && t->dims.size() == 1 && !t->data.empty(); };
    for (const auto& n : g.nodes) {
        if (n.op == "Conv" || n.op == "ConvTranspose") {
            Rec r; r.type = R_CONV; r.conv = convs.at(ci++); r.name = n.name;
            recs.push_back(r);
        } else if (n.op == "LayerNormalization") {
            if (n.inputs.size() < 3) throw Error("pack: LayerNormalization without scale/bias");
            Rec r; r.type = R_LN; r.a = g.find(n.inputs[1]); r.b = g.find(n.inputs[2]); r.name = n.name; r.eps = n.epsilon;
            if (!r.a || !r.b) throw Error("pack: LayerNormalization parameters are not initializers");
            recs.push_back(r);
        } else if (n.op == "Gemm" && n.inputs.size() >= 2) {
            const OnnxTensor* w = g.find(n.inputs[1]);
            if (w && w->dims.size() == 2 && !n.transA) {
                const OnnxTensor* wt = w;
                if (n.transB) {
                    const int N = (int)w->dims[0], K = (int)w->dims[1];
                    if ((size_t)N * K != w->data.size()) throw Error("pack: Gemm weight of '" + n.name + "' has no float data");
                    synth.emplace_back();
                    OnnxTensor& t = synth.back();
                    t.name = w->name + "^T";
                    t.dims = {K, N};
                    t.data.resize((size_t)K * N);
                    for (int nn = 0; nn < N; ++nn)
                        for (int k = 0; k < K; ++k) t.data[(size_t)k * N + nn] = w->data[(size_t)nn * K + k];
                    wt = &t;
                }
                Rec r; r.type = R_LIN; r.a = wt; r.name = n.name;
                r.b = n.inputs.size() > 2 && !n.inputs[2].empty() ? g.find(n.inputs[2]) : nullptr;
                recs.push_back(r);
                pendingLin = -1;
            }
        } else if (n.op == "Mul" && n.inputs.size() == 2) {
            // Mul(Div(...), gamma): second half of a decomposed LayerNorm
            for (int side = 0; side < 2; ++side) {
                const OnnxTensor* gamma = g.find(n.inputs[1 - side]);
                const OnnxNode* div = gi.producer(n.inputs[side]);
                if (!isVec(gamma) || !div || div->op != "Div" || div->inputs.size() != 2) continue;
                const OnnxNode* sq = gi.producer(div->inputs[1]);
                if (!sq || sq->op != "Sqrt") continue;
                float eps = 1e-5f;
                if (const OnnxNode* addEps = gi.producer(sq->inputs[0]))
                    if (addEps->op == "Add")
                        for (const auto& in : addEps->inputs)
                            if (const OnnxTensor* e = g.find(in))
                                if (e->data.size() == 1) eps = e->data[0];
                pendingLn.push_back({n.outputs.empty() ? std::string() : n.outputs[0], gamma, eps});
                break;
            }
        } else if (n.op == "MatMul" && n.inputs.size() == 2) {
            const OnnxTensor* w = g.find(n.inputs[1]);
            if (w && w->dims.size() == 2) {
                Rec r; r.type = R_LIN; r.a = w; r.name = n.name;
                recs.push_back(r);
                pendingLin = (int)recs.size() - 1;
                pendingOut = n.outputs.empty() ? "" : n.outputs[0];
            }
        } else if (n.op == "Add" && n.inputs.size() == 2) {
            const OnnxTensor* t = g.find(n.inputs[1]);
            const std::string other = n.inputs[0];
            if (!t) { t = g.find(n.inputs[0]); }
            if (!t) continue;
            bool wasLn = false;
            for (size_t k = 0; k < pendingLn.size(); ++k)
                if (isVec(t) && (n.inputs[0] == pendingLn[k].mulOut || n.inputs[1] == pendingLn[k].mulOut)) {
                    Rec r; r.type = R_LN; r.a = pendingLn[k].gamma; r.b = t; r.name = n.name; r.eps = pendingLn[k].eps;
                    recs.push_back(r);
                    pendingLn.erase(pendingLn.begin() + (long)k);
                    wasLn = true;
                    break;
                }
            if (wasLn) continue;
            if (t->dims.size() == 1 && pendingLin >= 0 && (n.inputs[0] == pendingOut || n.inputs[1] == pendingOut)) {
                recs[pendingLin].b = t;  // bias of the preceding MatMul
                pendingLin = -1;
            } else if (t->dims.size() >= 3 && t->dims[t->dims.size() - 1] == t->dims[t->dims.size() - 2]) {
                Rec r; r.type = R_ATTN; r.a = t; r.name = n.name;
                recs.push_back(r);
            }
        }
    }
    // pass 2: template  conv conv | blocks*L | down | blocks*L | down | blocks*3L | up | blocks*L | up | blocks*L | [up] | to_image
    size_t p = 0;
    auto need = [&](int type, const char* what) -> const Rec& {
        if (p >= recs.size() || recs[p].type != type) throw Error(std::string("pack: swin_unet template mismatch, expected ") + what + " at record " + std::to_string(p));
        return recs[p++];
    };
    const Rec& c0 = need(R_CONV, "patch conv 0");
    const Rec& c1 = need(R_CONV, "patch conv 1");
    if (c0.conv.cin != 3 || c0.conv.kh != 3 || c1.conv.kh != 3 || c1.conv.cin != c0.conv.cout || c0.conv.cout > 64 || c1.conv.cout % 32)
        throw Error("pack: unexpected swin_unet patch embedding");
    const int C = c1.conv.cout;
    m.dim = (uint32_t)C;
    m.layers.push_back(packLayer(c0.conv, false, 0, 64));   // 3 -> 64 stored channels (zero weights above cout)
    m.layers.push_back(packLayer(c1.conv, false, 64, 0));   // 64 stored -> C
    auto block = [&](int dim) {
        const Rec& n1 = need(R_LN, "norm1");
        const Rec& qkv = need(R_LIN, "qkv");
        const Rec& at = need(R_ATTN, "relative position bias");
        const Rec& pr = need(R_LIN, "proj");
        const Rec& n2 = need(R_LN, "norm2");
        const Rec& f1 = need(R_LIN, "mlp fc1");
        const Rec& f2 = need(R_LIN, "mlp fc2");
        auto ln = [&](const Rec& r) {
            if ((int)r.a->data.size() != dim || (int)r.b->data.size() != dim) throw Error("pack: LayerNorm width mismatch in " + r.name);
            PackedLayer L; L.name = r.name; L.kind = L_LN; L.cin = L.cout = (uint32_t)dim; L.eps = r.eps; L.gamma = r.a->data; L.beta = r.b->data;
            return L;
        };
        m.layers.push_back(ln(n1));
        PackedLayer q = packLinear(qkv.name, qkv.a, qkv.b, L_LINEAR);
        if ((int)q.cin != dim || (int)q.cout != 3 * dim) throw Error("pack: qkv shape mismatch in " + qkv.name);
        m.layers.push_back(q);
        {
            const auto& d = at.a->dims;
            const int nn = (int)d[d.size() - 1], heads = (int)d[d.size() - 3];
            int win = 1;
            while (win * win < nn) ++win;
            if (win * win != nn || dim % heads || (size_t)heads * nn * nn != at.a->data.size()) throw Error("pack: bad relative position bias in " + at.name);
            PackedLayer L; L.name = at.name; L.kind = L_ATTN; L.cin = L.cout = (uint32_t)dim; L.heads = (uint32_t)heads; L.window = (uint32_t)win; L.relpos = at.a->data;
            m.layers.push_back(L);
        }
        PackedLayer pj = packLinear(pr.name, pr.a, pr.b, L_LINEAR);
        if ((int)pj.cin != dim || (int)pj.cout != dim) throw Error("pack: proj shape mismatch in " + pr.name);
        m.layers.push_back(pj);
        m.layers.push_back(ln(n2));
        PackedLayer l1 = packLinear(f1.name, f1.a, f1.b, L_LINEAR), l2 = packLinear(f2.name, f2.a, f2.b, L_LINEAR);
        if ((int)l1.cin != dim || l2.cin != l1.cout || (int)l2.cout != dim) throw Error("pack: mlp shape mismatch in " + f1.name);
        m.layers.push_back(l1);
        m.layers.push_back(l2);
    };
    auto blocksUntil = [&](int dim) {  // consume blocks while the next record is a LayerNorm
        int nb = 0;
        while (p < recs.size() && recs[p].type == R_LN) { block(dim); ++nb; }
        if (nb == 0) throw Error("pack: swin stage without blocks");
        return nb;
    };
    auto down = [&](int cin, int cout) {
        const Rec& r = need(R_CONV, "patch down conv");
        if (r.conv.kh != 2 || r.conv.stride != 2 || r.conv.cin != cin || r.conv.cout != cout) throw Error("pack: unexpected PatchDown " + r.name);
        m.layers.push_back(packLayer(r.conv, false));
    };
    auto upl = [&](int cin, int cout) {
        const Rec& r = need(R_LIN, "patch up linear");
        PackedLayer L = packLinear(r.name, r.a, r.b, L_UPLIN);
        if ((int)L.cin != cin || (int)L.cout != cout) throw Error("pack: unexpected PatchUp " + r.name);
        m.layers.push_back(L);
    };
    blocksUntil(C);
    down(C, 2 * C);
    blocksUntil(2 * C);
    down(2 * C, 2 * C);
    blocksUntil(2 * C);
    upl(2 * C, 2 * C);
    blocksUntil(2 * C);
    upl(2 * C, C);
    blocksUntil(C);
    // [up0] to_image
    if (p + 2 == recs.size()) {
        upl(C, C);
        const Rec& r = need(R_LIN, "to_image");
        m.layers.push_back(packLinear(r.name, r.a, r.b, L_TOIMG, 0, 2));
        m.scale = 4;
    } else if (p + 1 == recs.size()) {
        const Rec& r = need(R_LIN, "to_image");
        const int N = (int)r.a->dims[1];
        m.scale = N == 3 ? 1 : 2;
        m.layers.push_back(packLinear(r.name, r.a, r.b, L_TOIMG, 0, (int)m.scale));
    } else {
        throw Error("pack: swin_unet template mismatch at the image head");
    }
    m.offset = 8 * m.scale;
    // what the shapes cannot tell: LeakyReLU(0.1) after both patch-embedding convs, the final clamp
    for (const Rec* r : {&c0, &c1}) {
        const OnnxNode* act = r->conv.node && !r->conv.node->outputs.empty() ? gi.consumerOp(r->conv.node->outputs[0], "LeakyRelu") : nullptr;
        if (!act || std::fabs(act->alpha - 0.1f) > 1e-6f) throw Error("pack: swin_unet patch embedding conv '" + r->name + "' is not followed by LeakyRelu(0.1)");
    }
    verifyClip01(g, "the swin_unet graph");
    return m;
}
}  // namespace

void composeUpToImage(const PackedLayer& U, const PackedLayer& L, std::vector<uint16_t>& wc, std::vector<float>& bc) {
    const int cmid = (int)U.cout, K = (int)U.ktot;
    if (U.kind != L_UPLIN || L.kind != L_TOIMG || L.upscale != 2 || (int)L.ktot != cmid || (int)U.npad != 4 * cmid || U.w.size() != (size_t)4 * cmid * K ||
        L.w.size() != (size_t)16 * cmid)
        throw Error("compose: PatchUp / ToImage shapes do not match");
    wc.assign((size_t)64 * K, 0);
    bc.assign(64, 0.f);
    std::vector<double> acc((size_t)K);
    for (int q0 = 0; q0 < 4; ++q0)
        for (int q1 = 0; q1 < 4; ++q1)
            for (int c3 = 0; c3 < 3; ++c3) {
                const int oy = 2 * (q0 >> 1) + (q1 >> 1), ox = 2 * (q0 & 1) + (q1 & 1);
                const int dst = (oy * 4 + ox) * 4 + c3, rowI = q1 * 4 + c3;
                std::fill(acc.begin(), acc.end(), 0.0);
                double b = L.bias[rowI];
                for (int c = 0; c < cmid; ++c) {
                    const double wi = halfBitsToFloat(L.w[(size_t)rowI * cmid + c]);
                    const uint16_t* urow = &U.w[(size_t)(q0 * cmid + c) * K];
                    for (int k = 0; k < K; ++k) acc[k] += wi * halfBitsToFloat(urow[k]);
                    b += wi * U.bias[q0 * cmid + c];
                }
                for (int k = 0; k < K; ++k) wc[(size_t)dst * K + k] = floatToHalfBits((float)acc[k]);
                bc[dst] = (float)b;
            }
}

bool isSwinGraph(const OnnxGraph& g) {
    // SwinUNet exports carry LayerNorm (fused, or decomposed into ... Sqrt -> Div -> Mul -> Add below opset 17) and an Erf GELU / Softmax;
    // the cunet family has none of these
    for (const auto& n : g.nodes)
        if (n.op == "LayerNormalization" || n.op == "Softmax" || n.op == "Erf") return true;
    return false;
}

PackedModel packFromOnnx(const OnnxGraph& g, int precision) {
    if (isSwinGraph(g)) {
        if (precision == W2X_PRECISION_TF32) throw Error("tf32 is not available for swin_unet models");
        return packSwin(g, precision);
    }
    std::vector<ConvNode> convs = collectConvs(g);
    PackedModel m;
    m.precision = (uint32_t)precision;
    for (size_t i = 0; i < convs.size(); ++i) {
        const ConvNode& c = convs[i];
        if (!c.transpose && c.kh == 1 && c.kw == 1) {
            // squeeze/excite pair: fc1 (C -> C/r) then fc2 (C/r -> C), attached to the previous layer
            if (m.layers.empty() || i + 1 >= convs.size()) throw Error("pack: dangling 1x1 conv " + c.name);
            const ConvNode& c2 = convs[i + 1];
            PackedLayer& L = m.layers.back();
            if (c2.transpose || c2.kh != 1 || c.cin != (int)L.cout || c2.cout != (int)L.cout || c2.cin != c.cout)
                throw Error("pack: 1x1 convs after " + L.name + " do not form a squeeze/excite block");
            L.se_r = (uint32_t)c.cout;
            L.se_w1.assign(c.w->data.begin(), c.w->data.end());   // [r][c][1][1]
            L.se_w2.assign(c2.w->data.begin(), c2.w->data.end()); // [c][r][1][1]
            L.se_b1.assign((size_t)c.cout, 0.f);
            L.se_b2.assign((size_t)c2.cout, 0.f);
            if (c.b) L.se_b1 = c.b->data;
            if (c2.b) L.se_b2 = c2.b->data;
            ++i;
            continue;
        }
        m.layers.push_back(packLayer(c, precision == W2X_PRECISION_TF32));
    }
    // template: UNet1 (8 layers) + UNet2 (14 layers), SURVEY 2.2
    const bool up = m.layers.size() > 7 && m.layers[7].kind == L_UP4;
    const std::vector<Expect> tmpl = {
        {L_CONV3, 4, 32, false},  {L_CONV3, 32, 64, false},  {L_DOWN2, 64, 64, false},   {L_CONV3, 64, 128, false},
        {L_CONV3, 128, 64, true}, {L_UP2, 64, 64, false},    {L_CONV3, 64, 64, false},   {up ? L_UP4 : L_CONV3, 64, 3, false},
        {L_CONV3, 4, 32, false},  {L_CONV3, 32, 64, false},  {L_DOWN2, 64, 64, false},   {L_CONV3, 64, 64, false},
        {L_CONV3, 64, 128, true}, {L_DOWN2, 128, 128, false}, {L_CONV3, 128, 256, false}, {L_CONV3, 256, 128, true},
        {L_UP2, 128, 128, false}, {L_CONV3, 128, 64, false}, {L_CONV3, 64, 64, true},    {L_UP2, 64, 64, false},
        {L_CONV3, 64, 64, false}, {L_CONV3, 64, 3, false}};
    if (m.layers.size() != tmpl.size())
        throw Error("pack: graph has " + std::to_string(m.layers.size()) + " convolution layers; the cunet template needs " +
                    std::to_string(tmpl.size()));
    for (size_t i = 0; i < tmpl.size(); ++i) {
        const PackedLayer& L = m.layers[i];
        if (L.kind != tmpl[i].kind || (int)L.cin != tmpl[i].cin || (int)L.cout != tmpl[i].cout || (L.se_r != 0) != tmpl[i].se)
            throw Error("pack: layer " + std::to_string(i) + " ('" + L.name + "') does not match the cunet template");
    }
    // ---- what the shapes cannot tell: activation slopes, skip crops, SE wiring, the final clamp ----
    {
        const GraphIndex gi(g);
        size_t li = 0;
        for (size_t i = 0; i < convs.size(); ++i) {
            const ConvNode& c = convs[i];
            const std::string out = c.node->outputs.empty() ? std::string() : c.node->outputs[0];
            if (!c.transpose && c.kh == 1 && c.kw == 1) {
                // SE: GlobalAveragePool -> 1x1 -> Relu -> 1x1 -> Sigmoid -> Mul
                const ConvNode& c2 = convs[i + 1];
                const OnnxNode* pool = gi.producer(c.node->inputs[0]);
                const bool pooled = pool && (pool->op == "GlobalAveragePool" || (pool->op == "ReduceMean" && pool->axes.size() == 2));
                if (!pooled) throw Error("pack: squeeze/excite '" + c.name + "' is not fed by a global average pool");
                if (!gi.consumerOp(out, "Relu")) throw Error("pack: squeeze/excite '" + c.name + "' is not followed by Relu");
                const OnnxNode* sg = gi.consumerOp(c2.node->outputs.empty() ? std::string() : c2.node->outputs[0], "Sigmoid");
                if (!sg || !gi.consumerOp(sg->outputs[0], "Mul")) throw Error("pack: squeeze/excite '" + c2.name + "' is not followed by Sigmoid -> Mul");
                ++i;
                continue;
            }
            const bool head = li == 7 || li == 21;
            const OnnxNode* act = gi.consumerOp(out, "LeakyRelu");
            if (head) {
                if (act) throw Error("pack: image head '" + c.name + "' has an activation (the kernels apply none)");
            } else {
                if (!act) throw Error("pack: conv '" + c.name + "' is not followed by LeakyRelu (the kernels fuse LeakyReLU(0.1))");
                if (std::fabs(act->alpha - 0.1f) > 1e-6f)
                    throw Error("pack: LeakyRelu after '" + c.name + "' has alpha " + std::to_string(act->alpha) + " (the kernels fuse 0.1)");
            }
            ++li;
        }
        std::vector<int> crops;
        for (const auto& n : g.nodes) {
            const int a = cropAmount(g, n);
            if (a > 0) crops.push_back(a);
        }
        std::sort(crops.begin(), crops.end());
        if (crops != std::vector<int>{4, 4, 16, 20})
            throw Error("pack: the skip-connection crops of the graph are not the cunet ones (4, 4, 16, 20)");
        int skipAdds = 0;
        for (const auto& n : g.nodes)
            if (n.op == "Add" && n.inputs.size() == 2 && !g.find(n.inputs[0]) && !g.find(n.inputs[1])) ++skipAdds;
        if (skipAdds != 4) throw Error("pack: expected 4 skip / residual additions in a cunet graph, found " + std::to_string(skipAdds));
        verifyClip01(g, "the cunet graph");
    }
    m.arch = up ? ARCH_UPCUNET : ARCH_CUNET;
    m.scale = up ? 2 : 1;
    m.offset = up ? 36 : 28;
    return m;
}

// ------------------------------------------------------------------------------------------------
// Flat file:  "W2XPACK2" | arch scale offset precision dim nlayers | per layer: header + blobs (4-byte aligned); the GEMM weight blob
// holds fp16 bits (precision FP16) or fp32 values (precision TF32)
// ------------------------------------------------------------------------------------------------
namespace {
void put32(std::vector<uint8_t>& o, uint32_t v) { for (int i = 0; i < 4; ++i) o.push_back((uint8_t)(v >> (8 * i))); }
template <class T>
void putVec(std::vector<uint8_t>& o, const std::vector<T>& v) {
    put32(o, (uint32_t)v.size());
    const size_t n = v.size() * sizeof(T);
    const size_t at = o.size();
    o.resize(at + ((n + 3) & ~size_t(3)), 0);
    if (n) std::memcpy(o.data() + at, v.data(), n);
}
struct In {
    const uint8_t* p; size_t n, i = 0;
    uint32_t u32() { if (i + 4 > n) throw Error("pack file truncated"); uint32_t v; std::memcpy(&v, p + i, 4); i += 4; return v; }
    template <class T> void vec(std::vector<T>& v) {
        const uint32_t cnt = u32();
        const size_t bytes = (size_t)cnt * sizeof(T), padded = (bytes + 3) & ~size_t(3);
        if (i + padded > n) throw Error("pack file truncated");
        v.resize(cnt);
        if (bytes) std::memcpy(v.data(), p + i, bytes);
        i += padded;
    }
};
}  // namespace

std::vector<uint8_t> serializePack(const PackedModel& m) {
    std::vector<uint8_t> o;
    const char magic[8] = {'W', '2', 'X', 'P', 'A', 'C', 'K', '2'};
    o.insert(o.end(), magic, magic + 8);
    put32(o, m.arch); put32(o, m.scale); put32(o, m.offset); put32(o, m.precision); put32(o, m.dim); put32(o, (uint32_t)m.layers.size());
    for (const auto& L : m.layers) {
        std::vector<char> nm(L.name.begin(), L.name.end());
        putVec(o, nm);
        put32(o, L.kind); put32(o, L.cin); put32(o, L.cout); put32(o, L.npad); put32(o, L.ktot); put32(o, L.taps); put32(o, L.se_r);
        put32(o, L.heads); put32(o, L.window); put32(o, L.upscale);
        uint32_t e; std::memcpy(&e, &L.eps, 4); put32(o, e);
        if (m.precision == W2X_PRECISION_TF32) putVec(o, L.wf);
        else putVec(o, L.w);
        putVec(o, L.bias); putVec(o, L.se_w1); putVec(o, L.se_b1); putVec(o, L.se_w2); putVec(o, L.se_b2);
        putVec(o, L.gamma); putVec(o, L.beta); putVec(o, L.relpos);
    }
    return o;
}

PackedModel deserializePack(const std::vector<uint8_t>& blob) {
    if (blob.size() < 32 || std::memcmp(blob.data(), "W2XPACK2", 8) != 0) throw Error("not a W2XPACK2 file");
    In in{blob.data(), blob.size(), 8};
    PackedModel m;
    m.arch = in.u32(); m.scale = in.u32(); m.offset = in.u32(); m.precision = in.u32(); m.dim = in.u32();
    const uint32_t nl = in.u32();
    if (nl > 4096) throw Error("pack file corrupt");
    m.layers.resize(nl);
    for (auto& L : m.layers) {
        std::vector<char> nm;
        in.vec(nm);
        L.name.assign(nm.begin(), nm.end());
        L.kind = in.u32(); L.cin = in.u32(); L.cout = in.u32(); L.npad = in.u32(); L.ktot = in.u32(); L.taps = in.u32(); L.se_r = in.u32();
        L.heads = in.u32(); L.window = in.u32(); L.upscale = in.u32();
        const uint32_t e = in.u32(); std::memcpy(&L.eps, &e, 4);
        if (m.precision == W2X_PRECISION_TF32) in.vec(L.wf);
        else in.vec(L.w);
        in.vec(L.bias); in.vec(L.se_w1); in.vec(L.se_b1); in.vec(L.se_w2); in.vec(L.se_b2);
        in.vec(L.gamma); in.vec(L.beta); in.vec(L.relpos);
        if (L.weightCount() != (size_t)L.npad * L.ktot || L.bias.size() != L.npad) throw Error("pack file: layer '" + L.name + "' has inconsistent sizes");
    }
    return m;
}

}  // namespace w2x
