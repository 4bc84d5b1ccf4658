// Host build of include/lgmi.h's lgmi_piece_ipc for tests/test_shard_split.py: its size and the offset of every
// field as the C++ compiler lays them out, to hold the ctypes mirror in l-giremi_b200/_lib.py to.  Test
// infrastructure; not part of the product library.
#include <cstddef>
#include <cstdint>
#include <cstring>

#include "../../include/lgmi.h"

#define FIELD(name) {#name, offsetof(lgmi_piece_ipc, name)}

static const struct {
  const char* name;
  size_t offset;
} kFields[] = {FIELD(plane_mem),   FIELD(dense_mem), FIELD(event),     FIELD(plane_word), FIELD(plane_words),
               FIELD(dense_off),   FIELD(dense_pairs), FIELD(batch_id), FIELD(unit),       FIELD(n_sites),
               FIELD(row_limit),   FIELD(ran),       FIELD(pid),       FIELD(pci_bus_id)};

extern "C" {
uint64_t piece_ipc_size() { return sizeof(lgmi_piece_ipc); }
// offset of the named field, or -1 if the struct has none of that name
int64_t piece_ipc_offset(const char* name) {
  for (const auto& f : kFields)
    if (!strcmp(f.name, name)) return (int64_t)f.offset;
  return -1;
}
}
