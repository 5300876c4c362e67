#include "pool.h"

#include <set>

namespace w2x {

EnginePool::EnginePool(const int* devices, int count) {
    if (!devices || count < 1 || count > 64) throw Error("engine pool: need 1..64 device ids");
    for (auto& s : state) s = FREE;
    for (int i = 0; i < count; ++i) {
        if (devices[i] < 0) throw Error("engine pool: negative device id");
        auto w = std::make_unique<Worker>();
        w->device = devices[i];
        workers.push_back(std::move(w));
    }
    for (auto& w : workers) w->th = std::thread([this, p = w.get()] { workerLoop(p); });
}

EnginePool::~EnginePool() {
    for (auto& w : workers) {
        {
            std::lock_guard<std::mutex> lk(w->mu);
            w->stop = true;
        }
        w->cv.notify_all();
    }
    for (auto& w : workers)
        if (w->th.joinable()) w->th.join();
}

void EnginePool::setMessageCallback(w2x_message_cb cb, void* user) {
    for (auto& w : workers) w->eng.impl.setMessageCallback(cb, user);
}

bool EnginePool::build(const std::string& onnxPath, const w2x_build_config& cfg) {
    // the artefact name hashes the device NAME (img2img_build.cpp:8-27): identical GPUs share one file
    std::set<std::string> done;
    for (auto& w : workers) {
        cudaDeviceProp prop{};
        if (cudaGetDeviceProperties(&prop, w->device) != cudaSuccess) {
            w->eng.impl.log(W2X_ERROR, "Failed to set cuda device to device id " + std::to_string(w->device) + ".", __FUNCTION__, __LINE__);
            return false;
        }
        if (!done.insert(prop.name).second) continue;
        w2x_build_config c = cfg;
        c.deviceId = w->device;
        if (!w->eng.impl.build(onnxPath, c)) return false;
    }
    return true;
}

bool EnginePool::load(const std::string& onnxPath, const w2x_render_config& cfg) {
    if (!sync()) return false;
    for (auto& w : workers) {
        w2x_render_config c = cfg;
        c.deviceId = w->device;
        if (!w->eng.impl.load(onnxPath, c)) return false;
    }
    return true;
}

int EnginePool::submit(const Frame& frame) {
    if (!frame.src || !frame.dst) return -1;
    return enqueue(Job{frame, 0});
}

int EnginePool::enqueue(Job job) {
    int ticket;
    {
        std::unique_lock<std::mutex> lk(stateMu);
        ticket = nextTicket;
        if (state[ticket % kRing] != FREE) return -1;  // kRing frames submitted and never waited for
        state[ticket % kRing] = QUEUED;
        ++nextTicket;
    }
    Worker& wk = *workers[ticket % workers.size()];
    {
        std::unique_lock<std::mutex> lk(wk.mu);
        wk.cv.wait(lk, [&] { return (int)wk.queue.size() < kQueueDepth || wk.stop; });  // back-pressure on the producer
        job.ticket = ticket;
        wk.queue.push_back(job);
    }
    wk.cv.notify_all();
    return ticket;
}

void EnginePool::finish(int ticket, bool ok) {
    {
        std::lock_guard<std::mutex> lk(stateMu);
        state[ticket % kRing] = ok ? DONE : FAILED;
    }
    stateCv.notify_all();
}

// One thread per device: enqueues up to three frames on its engine's copy / compute streams (Engine::submit) and retires them
// in order, so that the GPUs never wait for the thread that feeds the pool or for each other.
void EnginePool::workerLoop(Worker* w) {
    struct Flight { int engineTicket, ticket; };
    std::deque<Flight> flight;
    for (;;) {
        Job job{};
        bool have = false;
        {
            std::unique_lock<std::mutex> lk(w->mu);
            w->cv.wait(lk, [&] { return w->stop || !w->queue.empty() || !flight.empty(); });
            if (w->stop && w->queue.empty() && flight.empty()) return;
            if (!w->queue.empty() && flight.size() < 3) {
                job = w->queue.front();
                w->queue.pop_front();
                have = true;
            }
        }
        if (have) {
            w->cv.notify_all();  // a queue slot is free again
            const int t = w->eng.impl.submit(job.frame);
            if (t < 0) finish(job.ticket, false);
            else flight.push_back({t, job.ticket});
            continue;
        }
        if (!flight.empty()) {
            const Flight f = flight.front();
            flight.pop_front();
            finish(f.ticket, w->eng.impl.wait(f.engineTicket));
        }
    }
}

bool EnginePool::wait(int ticket) {
    std::unique_lock<std::mutex> lk(stateMu);
    if (ticket < 0 || ticket >= nextTicket || nextTicket - ticket > kRing) return false;
    State& s = state[ticket % kRing];
    if (s == FREE) return false;  // already consumed
    stateCv.wait(lk, [&] { return s == DONE || s == FAILED; });
    const bool ok = s == DONE;
    s = FREE;
    return ok;
}

bool EnginePool::sync() {
    std::unique_lock<std::mutex> lk(stateMu);
    stateCv.wait(lk, [&] {
        for (auto s : state)
            if (s == QUEUED) return false;
        return true;
    });
    return true;
}

}  // namespace w2x
