"""CPU test of the self-KV page accounting (csrc/kv_pager.h): a C++ driver compiled against the header with g++
checks page allocation, exhaustion, prompt sharing, the beam remap and the release of every page. A leaked or
doubly freed page would otherwise only show much later, as an exhausted pool or a wrong transcript."""
import os
import subprocess

from conftest import PKG

DRIVER = r"""
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "kv_pager.h"

namespace sw {
const char* last_error_string();
}
using namespace sw;

static int failures = 0;
#define CHECK(c)                                               \
  do {                                                         \
    if (!(c)) {                                                \
      fprintf(stderr, "line %d: CHECK(%s)\n", __LINE__, #c);   \
      ++failures;                                              \
    }                                                          \
  } while (0)

// every page is either free exactly once or held, with refc = the number of slot lists that hold it
static void check_consistent(const KvPager& pg, int n_slots) {
  std::vector<int> held(pg.refc.size(), 0), freed(pg.refc.size(), 0);
  for (int s = 0; s < n_slots; ++s)
    for (int i = 0; i < KV_MAX_PAGES; ++i)
      if (pg.page(s, i) >= 0) held[pg.page(s, i)]++;
  for (int p : pg.free_list) freed[p]++;
  for (size_t p = 0; p < held.size(); ++p) {
    CHECK(pg.refc[p] == held[p]);
    CHECK(freed[p] == (held[p] == 0 ? 1 : 0));
  }
}

static void release_all(KvPager& pg, int n_slots) {  // a remap of every slot onto itself with no positions
  std::vector<int> src(n_slots), copies, release;
  for (int s = 0; s < n_slots; ++s) src[s] = s;
  CHECK(pg.remap(0, src, 0, copies, release) == 0);
  CHECK(copies.empty());
  pg.unref(release);
  std::vector<int> fl = pg.free_list;
  std::sort(fl.begin(), fl.end());
  CHECK((int)fl.size() == (int)pg.refc.size());
  for (size_t i = 0; i < fl.size(); ++i) CHECK(fl[i] == (int)i);
}

int main() {
  KvPager pg;
  {  // ensure: one page per 32 positions; exhaustion is reported and changes nothing
    pg.reset(3, 2);
    for (int pos = 0; pos < 64; ++pos) CHECK(pg.ensure(0, pos) == 0);
    CHECK(pg.free_list.size() == 1 && pg.page(0, 0) >= 0 && pg.page(0, 1) >= 0 && pg.page(0, 2) < 0);
    CHECK(pg.ensure(1, 0) == 0 && pg.free_list.empty());
    const std::vector<int> owned = pg.owned, refc = pg.refc;
    CHECK(pg.ensure(0, 64) == -1);
    CHECK(strstr(last_error_string(), "self-KV page pool exhausted") != nullptr);
    CHECK(pg.owned == owned && pg.refc == refc && pg.free_list.empty());
    CHECK(pg.ensure(0, 63) == 0);  // a position whose page exists needs none
    int rows[KV_MAX_PAGES];
    pg.fill(0, rows);
    CHECK(rows[0] == pg.page(0, 0) && rows[1] == pg.page(0, 1) && rows[2] == 0 && rows[KV_MAX_PAGES - 1] == 0);
    check_consistent(pg, 2);
    release_all(pg, 2);
  }
  const int n_slots = 8;
  pg.reset(40, n_slots);
  {  // prompt sharing: a 40-token prompt of slot 1 into slots 1..5 (a window whose first slot is 1)
    for (int pos = 0; pos < 40; ++pos) CHECK(pg.ensure(1, pos) == 0);
    const int full = pg.page(1, 0), part = pg.page(1, 1);
    std::vector<int> copies, release;
    CHECK(pg.remap(1, std::vector<int>(5, 0), 40, copies, release) == 0);
    pg.unref(release);
    CHECK(pg.refc[full] == 5);
    CHECK(pg.page(1, 0) == full && pg.page(1, 1) == part && pg.refc[part] == 1);  // slot 1 keeps its own
    CHECK(copies.size() == 2 * 4);
    for (int j = 2; j <= 5; ++j) {
      CHECK(pg.page(j, 0) == full);
      const int c = pg.page(j, 1);
      CHECK(c >= 0 && c != part && pg.refc[c] == 1);
      CHECK(copies[2 * (j - 2)] == part && copies[2 * (j - 2) + 1] == c);
      CHECK(pg.page(j, 2) < 0);
    }
    check_consistent(pg, n_slots);
  }
  {  // beam permutation over slots 1..4 at 40 positions: src = {1, 1, 3, 3}
    std::vector<int> before(4);
    for (int j = 0; j < 4; ++j) before[j] = pg.page(1 + j, 1);
    const int full = pg.page(1, 0);
    const size_t n_free = pg.free_list.size();
    std::vector<int> copies, release;
    CHECK(pg.remap(1, {1, 1, 3, 3}, 40, copies, release) == 0);
    CHECK(pg.free_list.size() == n_free - 2);  // two fresh pages, nothing freed yet
    for (int p : before) CHECK(pg.refc[p] >= 1);
    CHECK(copies.size() == 2 * 2);
    CHECK(copies[0] == before[1] && copies[1] == pg.page(1, 1));  // slot 1 <- decoder 1's partial page
    CHECK(copies[2] == before[3] && copies[3] == pg.page(3, 1));  // slot 3 <- decoder 3's
    CHECK(pg.page(2, 1) == before[1] && pg.page(4, 1) == before[3]);  // src[j] == j keeps its own partial page
    for (int j = 1; j <= 4; ++j) CHECK(pg.page(j, 0) == full);
    CHECK(pg.page(5, 0) == full && pg.page(5, 1) >= 0);  // outside the window: untouched
    pg.unref(release);
    CHECK(pg.refc[full] == 5);
    CHECK(pg.refc[before[0]] == 0 && pg.refc[before[2]] == 0);  // the partial pages no decoder continues
    check_consistent(pg, n_slots);
  }
  {  // -1 leaves a slot as it is; a remap at a page boundary copies nothing
    for (int pos = 40; pos < 64; ++pos)
      for (int s = 1; s <= 5; ++s) CHECK(pg.ensure(s, pos) == 0);
    const int keep0 = pg.page(5, 0), keep1 = pg.page(5, 1), keep2 = pg.page(2, 1);
    const int old1 = pg.page(1, 1), old4 = pg.page(4, 1);
    std::vector<int> copies, release;
    CHECK(pg.remap(1, {3, -1, 0, 0, -1}, 64, copies, release) == 0);
    CHECK(copies.empty());
    CHECK(pg.page(5, 0) == keep0 && pg.page(5, 1) == keep1 && pg.page(2, 1) == keep2);
    CHECK(pg.page(1, 1) == old4 && pg.page(3, 1) == old1 && pg.page(4, 1) == old1);
    pg.unref(release);
    check_consistent(pg, n_slots);
  }
  release_all(pg, n_slots);
  if (failures) return 1;
  puts("ok");
  return 0;
}
"""


def test_kv_pager_accounting(tmp_path):
    csrc = os.path.join(PKG, "csrc")
    src = tmp_path / "kv_pager_driver.cpp"
    src.write_text(DRIVER)
    exe = tmp_path / "kv_pager_driver"
    subprocess.check_call(["g++", "-std=c++17", "-O1", "-Wall", "-Werror", "-I" + csrc, "-I/usr/local/cuda/include",
                           str(src), os.path.join(csrc, "errors.cpp"), "-o", str(exe)])
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    assert r.stdout.strip() == "ok"
