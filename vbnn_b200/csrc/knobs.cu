// knobs.cu -- see knobs.h.
#include "knobs.h"

#include <limits.h>
#include <stdlib.h>
#include <string.h>

#include <string>

namespace vbnn {

namespace {

struct Entry { const char* name; int Knobs::*field; };
const Entry kTable[] = {
    {"tc_bn", &Knobs::tc_bn},           {"tc_cg", &Knobs::tc_cg},         {"tc_gm", &Knobs::tc_gm},
    {"tc_clc", &Knobs::tc_clc},         {"tc_l2hint", &Knobs::tc_l2hint},         {"tc_staged", &Knobs::tc_staged}, {"tc_tacc", &Knobs::tc_tacc},
    {"tc_dw64", &Knobs::tc_dw64},       {"dw_eps16", &Knobs::dw_eps16},       {"lrt_split", &Knobs::lrt_split}, {"dw_split", &Knobs::dw_split},
    {"dp_overlap", &Knobs::dp_overlap}, {"no_graph", &Knobs::no_graph},   {"upd_bps", &Knobs::upd_bps},   {"peer_fused_push", &Knobs::peer_fused_push}, {"peer_transport", &Knobs::peer_transport}, {"peer_one_stream", &Knobs::peer_one_stream},
    {"peer_push_ctas", &Knobs::peer_push_ctas}, {"peer_wire_bf16", &Knobs::peer_wire_bf16},
    {"upd_coresident", &Knobs::upd_coresident},
};

// VBNN_<NAME>
bool from_env(const Entry& e, int* out) {
  std::string var = "VBNN_";
  for (const char* c = e.name; *c; ++c) var += (char)(*c >= 'a' && *c <= 'z' ? *c - 32 : *c);
  const char* v = getenv(var.c_str());
  if (!v || !*v) return false;
  *out = atoi(v);
  return true;
}

}  // namespace

Knobs& knobs() {
  static Knobs k = [] {
    Knobs k0;
    for (const Entry& e : kTable) {
      int v;
      if (from_env(e, &v)) k0.*(e.field) = v;
    }
    return k0;
  }();
  return k;
}

int knob_set(const char* name, int value) {
  if (!name) return -1;
  for (const Entry& e : kTable) {
    if (strcmp(e.name, name) != 0) continue;
    if (value == INT_MIN) {
      const Knobs def;
      int v = def.*(e.field);
      from_env(e, &v);
      value = v;
    }
    knobs().*(e.field) = value;
    return 0;
  }
  return -1;
}

int knob_get(const char* name, int* value) {
  if (!name || !value) return -1;
  for (const Entry& e : kTable)
    if (strcmp(e.name, name) == 0) { *value = knobs().*(e.field); return 0; }
  return -1;
}

}  // namespace vbnn
