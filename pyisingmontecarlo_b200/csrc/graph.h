// Host-side graph compiler: edge list -> CSR, coupling classification, torus recognition,
// greedy colouring.  Replaces the per-experiment adjacency build of GraphState::new
// (reference call site src/lattice.rs:199) with one compile per Lattice.
#pragma once
#include <stdint.h>

#include <string>
#include <vector>

namespace ising {

struct HostGraph {
    uint64_t nvars = 0;
    uint64_t nedges = 0;
    // explicit edge list (empty for implicit tori built by make_torus)
    std::vector<uint64_t> ea, eb;
    std::vector<double> ej;
    bool implicit_edges = false;

    std::vector<double> bias;  // nvars (all zero when !has_bias)
    bool has_bias = false;

    // CSR, neighbours ascending, ties in edge-list order (built on demand for implicit tori)
    bool csr_built = false;
    std::vector<uint64_t> row;
    std::vector<uint32_t> nbr;
    std::vector<double> jv;
    int max_degree = 0;

    bool integer_classes = false;  // all |J| equal (> 0) and no bias
    // uniform longitudinal field on a torus (ising_graph_torus_field): E gains - field * sum_i s_i;
    // the sweeps run the bit-sliced field kernel (sweep_field.cu), bias / has_bias stay unset
    bool field_graph = false;
    double field = 0.0;
    double jabs = 0.0;

    int kind = 0;  // ISING_KIND_*
    uint64_t dims[3] = {1, 1, 1};
    // stencil: bit d of fwd_sign[n] = 1 iff the bond n -> n + e_d has J > 0 (antiferro)
    std::vector<uint8_t> fwd_sign;
    bool uniform_sign = false;  // every bond has the same sign
    bool uniform_antiferro = false;

    int ncolors = 0;
    std::vector<uint32_t> color;  // general graphs only (stencil colour = parity of x+y+z)

    void build_csr();
    uint32_t color_of(uint64_t n) const;
    void edge_at(uint64_t e, uint64_t* a, uint64_t* b, double* j) const;
};

// Returns "" on success, else an error message.
std::string compile_from_edges(uint64_t nvars, uint64_t nedges, const uint64_t* a,
                               const uint64_t* b, const double* j, const double* biases,
                               HostGraph* out);
std::string make_torus(int dim, const uint64_t* L, double j0, int pmj, uint64_t j_seed,
                       HostGraph* out);

// Classes of edges that may be flipped as pairs in parallel (the two-spin "edge moves" of
// qmc GraphState::do_time_step, call sites src/lattice.rs:205, src/classicising.rs:100-106):
// a strong edge colouring - two edges of one class share no site and no bond joins them, so the
// energy change of one two-spin flip does not depend on another of the same class.
// Greedy in edge order; edges come out sorted by class.
struct EdgeClasses {
    std::vector<uint32_t> ea, eb;   // end points, class-sorted
    std::vector<uint32_t> eid;      // index in the edge list (Philox counter word 0)
    std::vector<float> wrel;        // |J_e| / max |J| (importance sampling of the edge choice)
    std::vector<uint32_t> off;      // nclasses + 1 offsets
};
void strong_edge_colouring(HostGraph* g, EdgeClasses* out);

// rand 0.8 SmallRng restated for Lattice::make_seeds (src/lattice.rs:83-91)
void make_seeds(uint64_t seed_gen, uint64_t n, uint64_t* out);

// src/lattice.rs:320-334 + 357-365; linear = documented interpolation instead of quirk Q1.
// Returns false when the reference would index out of bounds.
bool schedule_betas(const uint64_t* st, const double* sb, uint64_t n, uint64_t timesteps,
                    bool linear, double* out);

}  // namespace ising
