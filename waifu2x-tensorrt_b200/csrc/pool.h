// EnginePool: frame-parallel multi-GPU rendering inside ONE process (SURVEY 8e "frame-parallel": frame f -> GPU f mod N, a full weight
// replica and pinned-copy pipeline per GPU, one host worker thread per device, frames retired in order; no collective, no P2P).
// The reference is single-GPU (`--device`, /root/reference/src/main.cpp:70-74; cudaSetDevice at img2img_load.cpp:129): this is the
// "device list" extension of its operator surface, behind w2x_pool_* in include/w2x.h.
#pragma once
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "engine.h"

struct w2x_engine {
    w2x::Engine impl;
};

namespace w2x {

class EnginePool {
public:
    EnginePool(const int* devices, int count);
    ~EnginePool();
    EnginePool(const EnginePool&) = delete;
    EnginePool& operator=(const EnginePool&) = delete;

    int size() const { return (int)workers.size(); }
    w2x_engine* engine(int i) { return i >= 0 && i < size() ? &workers[i]->eng : nullptr; }
    void setMessageCallback(w2x_message_cb cb, void* user);
    bool build(const std::string& onnxPath, const w2x_build_config& cfg);   // once per distinct device name in the pool
    bool load(const std::string& onnxPath, const w2x_render_config& cfg);   // every engine, cfg.deviceId replaced by its own
    // frame `ticket` (0, 1, 2, ... in submission order) goes to engine ticket % size(); returns the ticket or -1.  A null image pointer is
    // refused here; the engine's other refusals (Engine::submit) fail the ticket's wait.
    int submit(const Frame& frame);
    bool wait(int ticket);   // true when that frame's dst is complete; tickets may be waited on in any order, each once
    bool sync();             // every submitted frame has been retired

private:
    struct Job { Frame frame; int ticket; };
    struct Worker {
        w2x_engine eng;
        int device = 0;
        std::thread th;
        std::mutex mu;
        std::condition_variable cv;
        std::deque<Job> queue;
        bool stop = false;
    };
    enum State : uint8_t { FREE = 0, QUEUED = 1, DONE = 2, FAILED = 3 };
    static constexpr int kRing = 256;      // tickets in flight (submitted, not yet waited for) must stay below this
    static constexpr int kQueueDepth = 4;  // frames a worker may hold beyond the engine's own three in flight

    int enqueue(Job job);   // assigns job.ticket
    void workerLoop(Worker* w);
    void finish(int ticket, bool ok);

    std::vector<std::unique_ptr<Worker>> workers;
    std::mutex stateMu;
    std::condition_variable stateCv;
    State state[kRing];
    int nextTicket = 0;
};

}  // namespace w2x
