// Concurrency stress of the native control-plane core, meant to be built with -fsanitize=thread and
// -fsanitize=address,undefined (tests/test_core_sanitizers.py; SURVEY.md §5.2 "race detection": the reference has
// no -race builds at all).  Exercises the same interleavings the Python layers produce: many producers / consumers on
// one rate-limited work queue, concurrent create / update / delete / watch on the store, expectation counters shared
// by workers, and the supervisor's spawn / kill / rename / reap paths.  Exit code 0 = invariants held.
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <set>
#include <thread>
#include <unistd.h>
#include <vector>

#include "store.h"
#include "supervisor.h"
#include "workqueue.h"

using namespace aitj;

#define CHECK(cond)                                                         \
  do {                                                                      \
    if (!(cond)) {                                                          \
      std::fprintf(stderr, "CHECK failed %s:%d: %s\n", __FILE__, __LINE__, #cond); \
      std::exit(1);                                                         \
    }                                                                       \
  } while (0)

static void stress_queue() {
  WorkQueue q("stress", 0.0005, 0.01, 1e6, 1000000);
  std::atomic<int> processed{0};
  std::mutex mu;
  std::set<std::string> in_flight;
  std::atomic<bool> overlap{false};
  std::vector<std::thread> ts;
  for (int c = 0; c < 4; ++c)
    ts.emplace_back([&] {
      for (;;) {
        auto k = q.get(0.2);
        if (!k) {
          if (q.shutting_down()) return;
          continue;
        }
        {
          std::lock_guard<std::mutex> lk(mu);
          if (!in_flight.insert(*k).second) overlap = true;      // a key is never handed to two workers at once
        }
        processed++;
        if (processed % 7 == 0) q.add_rate_limited(*k);
        else q.forget(*k);
        {
          std::lock_guard<std::mutex> lk(mu);
          in_flight.erase(*k);
        }
        q.done(*k);
      }
    });
  for (int p = 0; p < 4; ++p)
    ts.emplace_back([&, p] {
      for (int i = 0; i < 2000; ++i) {
        q.add("key-" + std::to_string((i * 7 + p) % 50));
        if (i % 5 == 0) q.add_after("late-" + std::to_string(i % 10), 0.001);
        if (i % 64 == 0) (void)q.len(), (void)q.len_waiting(), (void)q.num_requeues("key-1");
      }
    });
  for (size_t i = 4; i < ts.size(); ++i) ts[i].join();
  std::this_thread::sleep_for(std::chrono::milliseconds(100));
  q.shutdown();
  for (int i = 0; i < 4; ++i) ts[i].join();
  CHECK(!overlap.load());
  CHECK(processed.load() > 50);
}

static void stress_expectations() {
  Expectations e(300.0);
  std::vector<std::thread> ts;
  for (int t = 0; t < 4; ++t)
    ts.emplace_back([&] {
      for (int i = 0; i < 5000; ++i) {
        e.raise("job", 1, 1);
        (void)e.satisfied("job");
        e.lower("job", 1, 1);
        (void)e.peek("job");
      }
    });
  for (auto& t : ts) t.join();
  auto p = e.peek("job");
  CHECK(p && p->first == 0 && p->second == 0);
  CHECK(e.satisfied("job"));
}

static void stress_store() {
  Store s("", 4096);
  std::atomic<int> seen{0};
  std::atomic<bool> stop{false};
  std::vector<std::thread> ts;
  for (int w = 0; w < 2; ++w)
    ts.emplace_back([&] {
      int64_t id = s.watch_open("Pod", "", 0);
      while (!stop.load()) {
        auto ev = s.watch_next(id, 0.05);
        if (ev) seen++;
      }
      while (s.watch_next(id, 0.0)) seen++;
      s.watch_close(id);
    });
  for (int t = 0; t < 4; ++t)
    ts.emplace_back([&, t] {
      for (int i = 0; i < 400; ++i) {
        StoredObject o;
        o.kind = "Pod"; o.ns = "default"; o.name = "p-" + std::to_string(t) + "-" + std::to_string(i);
        o.uid = o.name; o.data = "{}"; o.labels["job"] = "j" + std::to_string(t);
        StoredObject c = s.create(o);
        c.data = "{\"v\":1}";
        bool conflict = false;
        try {
          s.update(c, c.rv + 1000);          // stale resourceVersion must be refused
        } catch (const StoreError& e) {
          conflict = e.reason == "Conflict";
        }
        CHECK(conflict);
        c = s.update(c, c.rv);
        (void)s.list("Pod", "default", {{"job", "j" + std::to_string(t)}});
        (void)s.get("Pod", "default", o.name);
        if (i % 2) s.remove("Pod", "default", o.name);
        if (i % 97 == 0) s.compact();
      }
    });
  for (size_t i = 2; i < ts.size(); ++i) ts[i].join();
  std::this_thread::sleep_for(std::chrono::milliseconds(100));
  stop = true;
  ts[0].join();
  ts[1].join();
  CHECK(s.count("Pod") == 4 * 200);
  CHECK(seen.load() > 0);
  CHECK(s.num_watchers() == 0);
}

// Owner index under concurrency: every thread creates jobs with dependents (some adopted later by an update, some
// handed to another owner, some deleted on their own), deletes the jobs and checks the cascade took exactly the
// dependents that belonged to it at that moment; a batched watcher drains every event in between.
static void stress_store_cascade() {
  Store s("", 1 << 16);
  std::atomic<bool> stop{false};
  std::atomic<long> events{0};
  // opened before any writer starts: a watch opened at "now" sees nothing published before it
  const int64_t id = s.watch_open("Pod", "", 0);
  std::thread watcher([&] {
    while (!stop.load()) events += static_cast<long>(s.watch_next_many(id, 0.02, 32).size());
    for (;;) {
      auto batch = s.watch_next_many(id, 0.0, 64, false);
      if (batch.empty()) break;
      events += static_cast<long>(batch.size());
    }
    s.watch_close(id);
  });
  std::vector<std::thread> ts;
  for (int t = 0; t < 4; ++t)
    ts.emplace_back([&, t] {
      for (int i = 0; i < 150; ++i) {
        const std::string tag = std::to_string(t) + "-" + std::to_string(i);
        StoredObject job;
        job.kind = "AITrainingJob"; job.ns = "ns"; job.name = "j-" + tag; job.uid = "uj-" + tag; job.data = "{}";
        s.create(job);
        StoredObject other = job;
        other.name = "o-" + tag; other.uid = "uo-" + tag;
        s.create(other);
        for (int k = 0; k < 4; ++k) {
          StoredObject pod;
          pod.kind = "Pod"; pod.ns = "ns"; pod.name = "p-" + tag + "-" + std::to_string(k);
          pod.uid = "up-" + tag + "-" + std::to_string(k); pod.data = "{}";
          if (k != 3) pod.owner_uids = {job.uid};            // k == 3 starts as an orphan
          s.create(pod);
        }
        StoredObject adopt = s.get("Pod", "ns", "p-" + tag + "-3");
        adopt.owner_uids = {job.uid};
        s.update(adopt, 0);                                   // adopted by the job
        StoredObject moved = s.get("Pod", "ns", "p-" + tag + "-0");
        moved.owner_uids = {other.uid};
        s.update(moved, 0);                                   // handed to the other owner
        s.remove("Pod", "ns", "p-" + tag + "-1");            // a dependent that goes on its own
        auto removed = s.remove("AITrainingJob", "ns", job.name);
        CHECK(removed.size() == 3);                           // the job, p-2 and the adopted p-3
        bool still = true;
        try { (void)s.get("Pod", "ns", "p-" + tag + "-0"); } catch (const StoreError&) { still = false; }
        CHECK(still);                                         // p-0 belongs to `other` now
        removed = s.remove("AITrainingJob", "ns", other.name);
        CHECK(removed.size() == 2);
      }
    });
  for (auto& t : ts) t.join();
  std::this_thread::sleep_for(std::chrono::milliseconds(50));
  stop = true;
  watcher.join();
  CHECK(s.count("Pod") == 0 && s.count("AITrainingJob") == 0);
  CHECK(events.load() == 4L * 150 * (4 + 2 + 4));             // per round: 4 ADDED, 2 MODIFIED, 4 DELETED pod events
  CHECK(s.num_watchers() == 0);
}

static void stress_supervisor() {
  Supervisor sup;
  std::map<std::string, std::string> env{{"PATH", "/usr/bin:/bin"}};
  std::atomic<int> exits{0};
  std::atomic<bool> stop{false};
  std::thread reaper([&] {
    const auto deadline = std::chrono::steady_clock::now() + std::chrono::seconds(60);
    while ((!stop.load() || exits.load() < 60) && std::chrono::steady_clock::now() < deadline) {
      for (auto& ev : sup.poll_exits(0.05)) {
        CHECK(ev.exit_code == 0 || ev.exit_code == 3 || ev.exit_code == 137);
        exits++;
      }
      if (stop.load() && sup.list().empty()) {
        // an exit that was reaped between the poll above and this check is queued but not counted yet
        for (auto& ev : sup.poll_exits(0.0)) {
          CHECK(ev.exit_code == 0 || ev.exit_code == 3 || ev.exit_code == 137);
          exits++;
        }
        break;
      }
    }
  });
  std::vector<std::thread> ts;
  for (int t = 0; t < 3; ++t)
    ts.emplace_back([&, t] {
      for (int i = 0; i < 20; ++i) {
        const std::string id = "c-" + std::to_string(t) + "-" + std::to_string(i);
        if (i % 3 == 0) {
          sup.spawn(id, {"/bin/sh", "-c", "exit 3"}, env, "", "", "", {});
        } else if (i % 3 == 1) {
          sup.spawn(id, {"/bin/sleep", "30"}, env, "", "", "", {});
          (void)sup.alive(id), (void)sup.pid_of(id);
          const std::string renamed = id + "-adopted";
          CHECK(sup.rename(id, renamed));
          CHECK(!sup.rename(id, renamed));
          sup.kill_proc(renamed, 9, true);
        } else {
          // re-keyed while it is already exiting: exactly one event, under whichever id won, and nothing left behind
          sup.spawn(id, {"/bin/true"}, env, "", "", "", {});
          (void)sup.rename(id, id + "-late");
        }
      }
    });
  for (auto& t : ts) t.join();
  stop = true;
  reaper.join();
  CHECK(exits.load() == 60);
  CHECK(sup.list().empty());
  // adoption of a process this supervisor did not spawn (agent-restart path)
  {
    pid_t pid = fork();
    if (pid == 0) {
      execl("/bin/sleep", "sleep", "30", static_cast<char*>(nullptr));
      _exit(127);
    }
    CHECK(pid > 0);
    setpgid(pid, pid);
    Supervisor sup2;
    sup2.adopt("adopted", pid);
    CHECK(sup2.alive("adopted") && sup2.pid_of("adopted") == pid);
    bool dup = false;
    try {
      sup2.adopt("adopted", pid);
    } catch (const SpawnError&) {
      dup = true;
    }
    CHECK(dup);
    sup2.kill_proc("adopted", 9, false);
    int got = 0;
    for (int i = 0; i < 100 && !got; ++i)
      for (auto& ev : sup2.poll_exits(0.05)) {
        CHECK(ev.id == "adopted" && ev.exit_code == 137);
        ++got;
      }
    CHECK(got == 1 && !sup2.alive("adopted"));
  }
  bool threw = false;
  try {
    sup.spawn("bad", {"/no/such/binary"}, env, "", "", "", {});
  } catch (const SpawnError&) {
    threw = true;
  }
  CHECK(threw);
}

int main() {
  stress_queue();
  stress_expectations();
  stress_store();
  stress_store_cascade();
  stress_supervisor();
  std::puts("core stress ok");
  return 0;
}
