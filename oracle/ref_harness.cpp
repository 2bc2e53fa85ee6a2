// TEST INFRASTRUCTURE ONLY — never linked into, imported by or executed from the product path.
//
// Headless C-ABI harness around the GENUINE reference class, compiled from the sources where they
// lie under $SPHSM_REFERENCE_DIR (see oracle/Makefile, target `ref`).  Nothing of the reference is copied
// into this repo: this file only #includes the reference header and calls the reference's own
// methods.  The resulting oracle/_ref/libsphsm_ref.so is (a) the pin for the C restatement in
// oracle/sphsm_oracle.c (bit-identical on every fixture, tests/test_oracle_vs_ref.py), (b) the
// generator of tests/golden/*.npz (tools/make_golden.py) and (c) the "reference" CPU baseline that
// bench.py times (cpu_baseline.kind == "reference").
//
// `#define private public` exposes the private tunables (World_Size, Max_Number_Paticles, ...) so
// the synthetic lattices (which need more than 50 000 particles / a world larger than 1.5^3) can be
// run through the unmodified reference arithmetic — SURVEY.md §8c describes exactly this trick.
#include <cstdio>
#include <cstring>
#include <cmath>
#include <vector>
#include <iostream>
#include <sstream>

#define private public
#include <SPH_SM_monodomain.h>
#undef private

namespace {
struct Quiet {  // the reference ctor/Init_Fluid print banners to cout; keep test logs clean
    std::streambuf *old;
    std::ostringstream sink;
    Quiet() : old(std::cout.rdbuf(sink.rdbuf())) {}
    ~Quiet() { std::cout.rdbuf(old); }
};
}  // namespace

extern "C" {

int ref_sizeof_particle() { return (int)sizeof(Particle); }

void *ref_create() {
    Quiet q;
    SPH_SM_monodomain *s = new SPH_SM_monodomain();
    // the reference never zero-initialises its duration accumulators (SURVEY §2 timers row)
    s->d_find_neighbors = s->d_corrected_velocity = s->d_intermediate_velocity = duration_d::zero();
    s->d_Density_SingPressure = s->d_cell_model = s->d_compute_Force = s->d_Update_Properties = duration_d::zero();
    return s;
}

void ref_destroy(void *h) { delete (SPH_SM_monodomain *)h; }

// Lift capacity / world for synthetic configs: re-derives exactly what the ctor derives from
// World_Size and Cell_Size (reference SPH_SM_monodomain.cpp:29-37, 51-52, 60-61).
void ref_resize(void *h, int max_particles, float wx, float wy, float wz) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    delete[] s->Particles;
    delete[] s->Cells;
    s->Max_Number_Paticles = max_particles;
    s->Number_Particles = 0;
    s->World_Size = m3Vector(wx, wy, wz);
    s->Grid_Size = s->World_Size / s->Cell_Size;
    s->Grid_Size.x = (int)ceil(s->Grid_Size.x);
    s->Grid_Size.y = (int)ceil(s->Grid_Size.y);
    s->Grid_Size.z = (int)ceil(s->Grid_Size.z);
    s->Number_Cells = (int)s->Grid_Size.x * (int)s->Grid_Size.y * (int)s->Grid_Size.z;
    s->Particles = new Particle[max_particles];
    s->Cells = new Cell[s->Number_Cells];
    s->bounds.min.zero();
    s->bounds.max.set(wx, wy, wz);
}

static std::vector<m3Vector> to_vec(const float *xyz, int n) {
    std::vector<m3Vector> v;
    v.reserve(n);
    for (int i = 0; i < n; i++) v.push_back(m3Vector(xyz[3 * i], xyz[3 * i + 1], xyz[3 * i + 2]));
    return v;
}

void ref_init_fluid(void *h, const float *xyz, int n) {
    Quiet q;
    ((SPH_SM_monodomain *)h)->Init_Fluid(to_vec(xyz, n));
}
void ref_stim_mesh(void *h, const float *xyz, int n) { ((SPH_SM_monodomain *)h)->turnOnStim_Mesh(to_vec(xyz, n)); }
void ref_stim_cube(void *h, const float *xyz, int n) { ((SPH_SM_monodomain *)h)->turnOnStim_Cube(to_vec(xyz, n)); }
void ref_set_stim(void *h, float cx, float cy, float cz, float radius, float strength) {
    ((SPH_SM_monodomain *)h)->set_stim(m3Vector(cx, cy, cz), radius, strength);
}
void ref_stim_off(void *h) { ((SPH_SM_monodomain *)h)->turnOffStim(); }
int ref_flip_quadratic(void *h) { return ((SPH_SM_monodomain *)h)->flip_quadratic(); }
int ref_flip_volume(void *h) { return ((SPH_SM_monodomain *)h)->flip_volume(); }
void ref_add_viscosity(void *h, float v) { ((SPH_SM_monodomain *)h)->add_viscosity(v); }

int ref_n(void *h) { return ((SPH_SM_monodomain *)h)->Get_Particle_Number(); }
void *ref_particles(void *h) { return ((SPH_SM_monodomain *)h)->Get_Paticles(); }
int ref_num_cells(void *h) { return ((SPH_SM_monodomain *)h)->Number_Cells; }

// stage ids follow the order of compute_SPH_SM_monodomain (reference cpp:794-824); 0 = whole step
void ref_stage(void *h, int stage) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    switch (stage) {
        case 0: s->Animation(); break;
        case 1: s->Find_neighbors(); break;
        case 2: s->calculate_corrected_velocity(); break;
        case 3: s->calculate_intermediate_velocity(); break;
        case 4: s->Compute_Density_SingPressure(); break;
        case 5: s->calculate_cell_model(); break;
        case 6: s->Compute_Force(); break;
        case 7: s->Update_Properties(); break;
        default: break;
    }
}

void ref_steps(void *h, int n) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    for (int i = 0; i < n; i++) s->Animation();
}

// scalar parameters as the reference computed them: K, Stand_Density, Time_Delta, mu, Poly6, Spiky,
// B_spline, sigma, alpha, beta, kernel, stim_strength, velocity_mixing, Wall_Hit, Cm, Beta
void ref_constants(void *h, float *out16) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    float v[16] = {s->K, s->Stand_Density, s->Time_Delta, s->mu, s->Poly6_constant, s->Spiky_constant,
                   s->B_spline_constant, s->sigma, s->alpha, s->beta, s->kernel, s->stim_strength,
                   s->velocity_mixing, s->Wall_Hit, s->Cm, s->Beta};
    memcpy(out16, v, sizeof(v));
}

// bucket contents after Find_neighbors: CSR over cells with particle indices in bucket order
// (reference cpp:199-213).  Returns total entries; pass NULL to query sizes only.
int ref_cells_csr(void *h, int *cell_start /*cells+1*/, int *indices /*n*/) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    int tot = 0;
    for (int c = 0; c < s->Number_Cells; c++) {
        if (cell_start) cell_start[c] = tot;
        for (Particle *p : s->Cells[c].contained_particles) {
            if (indices) indices[tot] = (int)(p - s->Particles);
            tot++;
        }
    }
    if (cell_start) cell_start[s->Number_Cells] = tot;
    return tot;
}

int ref_cell_hash(void *h, float x, float y, float z) {
    SPH_SM_monodomain *s = (SPH_SM_monodomain *)h;
    return s->Calculate_Cell_Hash(s->Calculate_Cell_Position(m3Vector(x, y, z)));
}

float ref_poly6(void *h, float r2) { return ((SPH_SM_monodomain *)h)->Poly6(r2); }
float ref_spiky(void *h, float r) { return ((SPH_SM_monodomain *)h)->Spiky(r); }
float ref_visco(void *h, float r) { return ((SPH_SM_monodomain *)h)->Visco(r); }
float ref_bspline2(void *h, float r) { return ((SPH_SM_monodomain *)h)->B_spline_2(r); }

// small-matrix KATs for the restatement (m3Matrix.cpp:73-113, m3Matrix.h:293-318, m9Matrix.cpp:80-102)
void ref_polar3(const float *a9, float *r9) {
    m3Matrix A, R, S;
    memcpy(&A.r00, a9, 9 * sizeof(float));
    m3Matrix::polarDecomposition(A, R, S);
    memcpy(r9, &R.r00, 9 * sizeof(float));
}
int ref_invert3(float *a9) {
    m3Matrix A;
    memcpy(&A.r00, a9, 9 * sizeof(float));
    bool ok = A.invert();
    memcpy(a9, &A.r00, 9 * sizeof(float));
    return ok ? 1 : 0;
}
void ref_invert9(float *a81) {
    m9Matrix A;
    memcpy(&A.r00, a81, 81 * sizeof(float));
    A.invert();
    memcpy(a81, &A.r00, 81 * sizeof(float));
}

}  // extern "C"
