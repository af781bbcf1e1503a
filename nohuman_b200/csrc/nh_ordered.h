/* nh_ordered.h — an ordered work queue for the file pipeline's stages.
 *
 * Items leave in the order they entered, whatever order the workers finish them in, and at most `window`
 * items are inside at once, so a slow consumer holds back the producer instead of letting memory grow.
 * Inside, an item is queued (waiting for a worker), claimed (a worker or the pusher has it) or done (the
 * consumer may take it once everything before it has left).
 *
 * Host-only on purpose: no CUDA header, so that a plain C++ test can build it. */
#ifndef NH_ORDERED_H
#define NH_ORDERED_H

#include <stddef.h>

#include <algorithm>
#include <condition_variable>
#include <deque>
#include <memory>
#include <mutex>
#include <vector>

template <typename T>
class OrderedQueue {
 public:
  typedef std::shared_ptr<T> Ptr;
  enum State { QUEUED, CLAIMED, DONE };

  explicit OrderedQueue(size_t window) : window_(window) {}

  /* enters `item` behind everything pushed before it, waiting while the window is full; false, with the
   * item not entered, once the queue is closed or stopped */
  bool push(Ptr item, State state) {
    std::unique_lock<std::mutex> lk(m_);
    space_.wait(lk, [&] { return slots_.size() < window_ || closed_ || stopped_; });
    if (closed_ || stopped_) return false;
    slots_.push_back(Slot{std::move(item), state});
    if (state == QUEUED) work_.notify_one();
    if (state == DONE && slots_.size() == 1) ready_.notify_all();
    return true;
  }

  /* the oldest queued item, now claimed; null once stopped, or once closed with nothing queued */
  Ptr take() {
    std::unique_lock<std::mutex> lk(m_);
    auto it = wait_queued(lk);
    if (it == slots_.end()) return nullptr;
    it->state = CLAIMED;
    return it->item;
  }

  /* from the oldest queued item on, the longest run of consecutive queued items whose size(item) add up to
   * at most `limit`, and always at least one item, all claimed; empty when take() would return null */
  template <typename Size>
  std::vector<Ptr> take(size_t limit, Size size) {
    std::vector<Ptr> run;
    std::unique_lock<std::mutex> lk(m_);
    size_t total = 0;
    for (auto it = wait_queued(lk); it != slots_.end() && it->state == QUEUED; ++it) {
      const size_t n = size(*it->item);
      if (!run.empty() && total + n > limit) break;
      total += n;
      it->state = CLAIMED;
      run.push_back(it->item);
    }
    return run;
  }

  /* marks a claimed item, or every item of a batch, done */
  void done(const Ptr &item) {
    std::lock_guard<std::mutex> lk(m_);
    mark_done(item);
  }
  void done(const std::vector<Ptr> &items) {
    std::lock_guard<std::mutex> lk(m_);
    for (const Ptr &item : items) mark_done(item);
  }

  /* the front item once it is done, out of the queue; null once stopped, or once closed and empty */
  Ptr pop() {
    std::unique_lock<std::mutex> lk(m_);
    ready_.wait(lk, [&] { return stopped_ || (closed_ && slots_.empty()) || (!slots_.empty() && slots_.front().state == DONE); });
    if (stopped_ || slots_.empty()) return nullptr;
    Ptr item = std::move(slots_.front().item);
    slots_.pop_front();
    space_.notify_one();
    return item;
  }

  /* no more pushes: workers and the consumer still finish everything inside */
  void close() {
    std::lock_guard<std::mutex> lk(m_);
    closed_ = true;
    wake_all();
  }

  /* abandon: every blocked or later push, take and pop returns at once */
  void stop() {
    std::lock_guard<std::mutex> lk(m_);
    stopped_ = true;
    wake_all();
  }

 private:
  struct Slot {
    Ptr item;
    State state;
  };

  /* the oldest queued slot, waiting for one while the queue is open; end() when there will be none */
  auto wait_queued(std::unique_lock<std::mutex> &lk) {
    auto first = slots_.end();
    work_.wait(lk, [&] {
      if (stopped_) return true;
      first = std::find_if(slots_.begin(), slots_.end(), [](const Slot &s) { return s.state == QUEUED; });
      return first != slots_.end() || closed_;
    });
    return stopped_ ? slots_.end() : first;
  }
  void mark_done(const Ptr &item) {
    for (Slot &s : slots_)
      if (s.item == item) s.state = DONE;
    if (!slots_.empty() && slots_.front().state == DONE) ready_.notify_all();
  }
  void wake_all() {
    space_.notify_all();
    work_.notify_all();
    ready_.notify_all();
  }

  std::mutex m_;
  std::condition_variable space_, work_, ready_; /* pushers, takers, the consumer */
  std::deque<Slot> slots_;                       /* entry order */
  size_t window_;
  bool closed_ = false, stopped_ = false;
};

#endif
