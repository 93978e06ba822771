// Self-KV page bookkeeping (host): the page list of every decoder slot over the engine's page pool, with
// reference counts, so that decoders sharing a prefix share its full pages. Plain C++: the device sees the
// pages only through the page list each step row carries (DecRow::pages, filled by fill()).
#pragma once
#include <algorithm>
#include <vector>

#include "host_common.h"
#include "kernels.cuh"

namespace sw {

struct KvPager {
  std::vector<int> owned;      // [slot][KV_MAX_PAGES]: page id, or -1
  std::vector<int> refc;       // per page: slots whose list holds it
  std::vector<int> free_list;  // pages with refc 0, taken from the back

  void reset(int n_pages, int n_slots) {
    refc.assign(n_pages, 0);
    free_list.resize(n_pages);
    for (int i = 0; i < n_pages; ++i) free_list[i] = n_pages - 1 - i;
    owned.assign((size_t)n_slots * KV_MAX_PAGES, -1);
  }
  int page(int slot, int i) const { return owned[(size_t)slot * KV_MAX_PAGES + i]; }

  // make sure `slot` has a page for position pos; on -1 the pool is exhausted and nothing changed
  int ensure(int slot, int pos) {
    int& p = owned[(size_t)slot * KV_MAX_PAGES + pos / KV_PAGE];
    if (p < 0) p = alloc();
    return p < 0 ? -1 : 0;
  }

  // Positions [0, n_kv) of slot slot0 + src[j] become slot slot0 + j's, for every j with src[j] >= 0 (the other
  // slots keep theirs). Full pages are shared by reference; the partly filled last page is copied unless the slot
  // continues its own sequence. Appends the (source, copy) page pairs to `copies` and the slots' previous pages to
  // `release`: a copy may read a page only the release frees, so unref(release) follows the copies' enqueue.
  int remap(int slot0, const std::vector<int>& src, int n_kv, std::vector<int>& copies, std::vector<int>& release) {
    const int n = (int)src.size(), np = (n_kv + KV_PAGE - 1) / KV_PAGE;
    std::vector<int> next((size_t)n * KV_MAX_PAGES, -1);  // every new list first: a source may be a destination
    for (int j = 0; j < n; ++j) {
      if (src[j] < 0) continue;
      for (int i = 0; i < np; ++i) {
        const int sp = page(slot0 + src[j], i);
        int& dp = next[(size_t)j * KV_MAX_PAGES + i];
        if ((i + 1) * KV_PAGE <= n_kv || src[j] == j) {
          ++refc[sp];
          dp = sp;
        } else {
          if ((dp = alloc()) < 0) return -1;
          copies.push_back(sp);
          copies.push_back(dp);
        }
      }
    }
    for (int j = 0; j < n; ++j) {
      if (src[j] < 0) continue;
      int* own = &owned[(size_t)(slot0 + j) * KV_MAX_PAGES];
      for (int i = 0; i < KV_MAX_PAGES; ++i) {
        if (own[i] >= 0) release.push_back(own[i]);
        own[i] = next[(size_t)j * KV_MAX_PAGES + i];
      }
    }
    return 0;
  }
  void unref(const std::vector<int>& pages) {
    for (int p : pages)
      if (--refc[p] == 0) free_list.push_back(p);
  }

  // the page list of a step row (DecRow::pages): 0 for an entry the slot has no page for
  void fill(int slot, int* pages) const {
    for (int i = 0; i < KV_MAX_PAGES; ++i) pages[i] = std::max(0, page(slot, i));
  }

 private:
  int alloc() {
    if (free_list.empty()) {
      set_last_error("self-KV page pool exhausted");
      return -1;
    }
    const int p = free_list.back();
    free_list.pop_back();
    refc[p] = 1;
    return p;
  }
};

}  // namespace sw
