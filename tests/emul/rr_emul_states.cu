// rr_emul_states.cu — HOST execution of rr_save_states / rr_load_states: rr_emul.cu plus three exports.
//
// TEST INFRASTRUCTURE ONLY, built into its own test library (tests/emul/emul_states.py).  The loops below run the row
// layout and the index rules of the kernels k_save_rows / k_load_rows (rr_sim.cuh row_unit_get / row_unit_put,
// save_source / load_source) on EmulBatch columns plus a start array [3R + 2B][N], so that the CPU tier checks the byte
// layout, the skip rules for out-of-range indices and the continuation of a loaded state without a GPU.
#include "rr_emul.cu"

static RowLayout layout_of(const rr_config *cfg) { return row_layout(EMUL_DISPATCH(cfg, columns_t), cfg->observer); }

extern "C" {

// rr_snapshot_bytes_per_env
int64_t emul_row_bytes(const rr_config *cfg) { return layout_of(cfg).bytes(); }

// rr_save_states on host columns: rows [m][S] bytes; env NULL: env j
void emul_save_rows(const rr_config *cfg, const uint64_t *sf, const uint64_t *start, const uint32_t *si, int64_t N,
                    const int64_t *env, int64_t m, uint64_t *rows) {
  const RowLayout L = layout_of(cfg);
  for (int64_t j = 0; j < m; j++) {
    const int64_t e = save_source(env, j, N);
    if (e < 0) continue;
    for (int u = 0; u < L.units(); u++) rows[j * L.units() + u] = row_unit_get(L, sf, start, si, N, e, u);
  }
}

// rr_load_states on host columns; slot NULL: row i
void emul_load_rows(const rr_config *cfg, const uint64_t *rows, int64_t m, const int64_t *slot, int64_t N, uint64_t *sf,
                    uint64_t *start, uint32_t *si) {
  const RowLayout L = layout_of(cfg);
  for (int64_t i = 0; i < N; i++) {
    const int64_t r = load_source(slot, i, m);
    if (r < 0) continue;
    for (int u = 0; u < L.units(); u++) row_unit_put(L, sf, start, si, N, i, u, rows[r * L.units() + u]);
  }
}
}
