/* Checks nohuman_b200/csrc/nh_ordered.h (the file pipeline's ordered work queue) on the host, built with
 * ThreadSanitizer by tests/test_ordered_queue.py.  Prints "OK" and exits 0 when every check holds. */
#include <stdio.h>
#include <stdlib.h>

#include <atomic>
#include <chrono>
#include <mutex>
#include <random>
#include <thread>
#include <vector>

#include "../../nohuman_b200/csrc/nh_ordered.h"

static std::atomic<int> failures{0};
#define CHECK(cond)                                                     \
  do {                                                                  \
    if (!(cond)) {                                                      \
      fprintf(stderr, "%s:%d: CHECK(%s) failed\n", __FILE__, __LINE__, #cond); \
      failures++;                                                       \
    }                                                                   \
  } while (0)

struct Item {
  long seq = 0;      /* entry order */
  int pusher = 0;
  long pusher_seq = 0;
  size_t size = 0;
  long value = -1;   /* written by whoever finishes the item */
};
typedef OrderedQueue<Item> Q;
typedef std::shared_ptr<Item> P;

static void pause_us(std::mt19937 &rng, int max_us) {
  std::this_thread::sleep_for(std::chrono::microseconds(rng() % (unsigned)(max_us + 1)));
}

static P item(long seq, size_t size = 1) {
  auto p = std::make_shared<Item>();
  p->seq = seq;
  p->size = size;
  return p;
}

/* Several pushers (entering queued, claimed or done items), single and batch takers, one consumer, random
 * delays everywhere.  With `ordered_entry` the pushers enter under a lock that also numbers the items, the
 * way the pipeline's classifiers enter Works, so pop order must be exactly that numbering; without it, each
 * pusher's own items must still pop in its order. */
static void stress(bool ordered_entry) {
  const size_t window = 8, limit = 5;
  const int pushers = 3, workers = 3, batch_workers = 2, per_pusher = 400;
  Q q(window);
  std::mutex entry_m;
  long next_seq = 0;
  std::atomic<long> in{0}, out{0}, max_inside{0};
  std::atomic<int> pushers_left{pushers};
  std::vector<std::thread> ts;
  for (int p = 0; p < pushers; p++)
    ts.emplace_back([&, p] {
      std::mt19937 rng(100 + p);
      for (long k = 0; k < per_pusher; k++) {
        const int r = (int)(rng() % 10);
        const Q::State st = r < 6 ? Q::QUEUED : r < 8 ? Q::CLAIMED : Q::DONE;
        P it = item(0, 1 + rng() % 3);
        it->pusher = p;
        it->pusher_seq = k;
        if (st == Q::DONE) it->value = k;
        {
          std::unique_lock<std::mutex> lk(entry_m, std::defer_lock);
          if (ordered_entry) {
            lk.lock();
            it->seq = next_seq++;
          }
          CHECK(q.push(it, st));
        }
        /* `out` counts a pop before it happens, so in - out never exceeds what is inside */
        const long inside = ++in - out.load();
        CHECK(inside <= (long)window);
        long m = max_inside.load();
        while (inside > m && !max_inside.compare_exchange_weak(m, inside)) {
        }
        if (st == Q::CLAIMED) {
          pause_us(rng, 50);
          it->value = k;
          q.done(it);
        }
        pause_us(rng, 20);
      }
      if (--pushers_left == 0) q.close();
    });
  for (int w = 0; w < workers; w++)
    ts.emplace_back([&, w] {
      std::mt19937 rng(200 + w);
      while (P it = q.take()) {
        pause_us(rng, 100);
        it->value = it->pusher_seq;
        q.done(it);
      }
    });
  for (int w = 0; w < batch_workers; w++)
    ts.emplace_back([&, w] {
      std::mt19937 rng(300 + w);
      for (;;) {
        std::vector<P> run = q.take(limit, [](const Item &i) { return i.size; });
        if (run.empty()) break;
        size_t total = 0;
        for (size_t i = 0; i < run.size(); i++) {
          total += run[i]->size;
          if (ordered_entry && i) CHECK(run[i]->seq == run[i - 1]->seq + 1); /* consecutive entries */
        }
        CHECK(run.size() == 1 || total <= limit);
        pause_us(rng, 150);
        for (P &it : run) it->value = it->pusher_seq;
        q.done(run);
      }
    });
  std::mt19937 rng(400);
  long popped = 0, next_of[pushers] = {0};
  for (;;) {
    out++;
    P it = q.pop();
    if (!it) break;
    if (ordered_entry) CHECK(it->seq == popped);
    CHECK(it->pusher_seq == next_of[it->pusher]);
    next_of[it->pusher] = it->pusher_seq + 1;
    CHECK(it->value == it->pusher_seq); /* finished before it left */
    popped++;
    if (popped % 50 == 0) /* a stalled consumer: the pushers fill the window and wait */
      std::this_thread::sleep_for(std::chrono::milliseconds(2));
    else
      pause_us(rng, 30);
  }
  for (auto &t : ts) t.join();
  CHECK(popped == (long)pushers * per_pusher);
  CHECK(max_inside.load() == (long)window); /* the window was filled */
}

/* take(limit, size): the run starts at the oldest queued item, stops at the first item that is not queued
 * or would pass the limit, and holds at least one item even when that one alone passes it. */
static void batch_take() {
  Q q(16);
  std::vector<P> v;
  const size_t sizes[] = {4, 3, 3, 2, 9, 1, 1, 1};
  const Q::State states[] = {Q::DONE, Q::QUEUED, Q::QUEUED, Q::QUEUED, Q::QUEUED, Q::CLAIMED, Q::QUEUED, Q::QUEUED};
  for (int i = 0; i < 8; i++) {
    v.push_back(item(i, sizes[i]));
    CHECK(q.push(v.back(), states[i]));
  }
  auto size = [](const Item &i) { return i.size; };
  std::vector<P> r = q.take(6, size); /* 3 + 3 */
  CHECK(r.size() == 2 && r[0] == v[1] && r[1] == v[2]);
  r = q.take(1, size); /* 2 alone passes 1: still one item */
  CHECK(r.size() == 1 && r[0] == v[3]);
  r = q.take(100, size); /* stops before the claimed item */
  CHECK(r.size() == 1 && r[0] == v[4]);
  r = q.take(100, size); /* skips the claimed item */
  CHECK(r.size() == 2 && r[0] == v[6] && r[1] == v[7]);
  q.close(); /* nothing queued, and nothing will be */
  CHECK(q.take() == nullptr && q.take(100, size).empty());
  /* pop: only a done front leaves; v[5] was entered claimed and blocks everything behind it */
  CHECK(q.pop() == v[0]);
  q.done({v[1], v[2], v[3], v[4], v[6], v[7]});
  std::atomic<bool> got{false};
  std::thread t([&] {
    CHECK(q.pop() == v[1]);
    CHECK(q.pop() == v[2]);
    CHECK(q.pop() == v[3]);
    CHECK(q.pop() == v[4]);
    CHECK(q.pop() == v[5]);
    got = true;
  });
  std::this_thread::sleep_for(std::chrono::milliseconds(50));
  CHECK(!got.load());
  q.done(v[5]);
  t.join();
  CHECK(got.load());
  CHECK(q.pop() == v[6] && q.pop() == v[7] && q.pop() == nullptr);
}

/* close(): no more pushes, but everything inside is still taken, finished and popped in order */
static void close_drains() {
  Q q(4);
  std::vector<P> v;
  for (int i = 0; i < 4; i++) {
    v.push_back(item(i));
    CHECK(q.push(v.back(), i == 2 ? Q::DONE : Q::QUEUED));
  }
  q.close();
  CHECK(!q.push(item(9), Q::QUEUED));
  std::thread worker([&] {
    while (P it = q.take()) {
      it->value = it->seq;
      q.done(it);
    }
  });
  for (int i = 0; i < 4; i++) {
    P it = q.pop();
    CHECK(it == v[i]);
    if (i != 2 && it) CHECK(it->value == i);
  }
  CHECK(q.pop() == nullptr);
  worker.join();
}

/* stop() releases a push blocked on a full window, a take with nothing queued and a pop whose front is not
 * done, and later calls return at once */
static void stop_releases() {
  Q q(2);
  CHECK(q.push(item(0), Q::CLAIMED));
  CHECK(q.push(item(1), Q::CLAIMED));
  std::atomic<int> returned{0};
  bool pushed = true;
  P taken = item(7), popped = item(7);
  std::thread tp([&] {
    pushed = q.push(item(2), Q::QUEUED);
    returned++;
  });
  std::thread tt([&] {
    taken = q.take();
    returned++;
  });
  std::thread to([&] {
    popped = q.pop();
    returned++;
  });
  std::this_thread::sleep_for(std::chrono::milliseconds(100));
  CHECK(returned.load() == 0); /* all three are blocked */
  q.stop();
  tp.join();
  tt.join();
  to.join();
  CHECK(returned.load() == 3);
  CHECK(!pushed && taken == nullptr && popped == nullptr);
  CHECK(!q.push(item(3), Q::DONE) && q.take() == nullptr && q.pop() == nullptr);
}

int main() {
  stress(true);
  stress(false);
  batch_take();
  close_drains();
  stop_releases();
  if (failures) {
    fprintf(stderr, "%d check(s) failed\n", failures.load());
    return 1;
  }
  printf("OK\n");
  return 0;
}
