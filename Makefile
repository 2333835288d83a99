# Build recipe for libb200nb (the product), the oracle (test infrastructure) and the reference-side binaries.
# `python -c "import __graft_entry__ as g; g.build()"` runs the same commands.
NVCC      ?= nvcc
CXX       ?= g++
# the image exports CC=/opt/gcc/bin/gcc, which has no libgomp.spec: use the distro compiler for the OpenMP oracle
ORACLE_CC ?= $(shell command -v /usr/bin/gcc || echo gcc)
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC
PKG       := nbody-eurohpc_b200
LIB       := $(PKG)/b200nb/libb200nb.so
REF       ?= /root/reference

all: lib oracle field_oracle neighbors_oracle fof_oracle groups_oracle tracers_oracle tidal_oracle components_oracle external_oracle phase_fof_oracle scf_oracle

# the default force-kernel variant with its hot loop re-ordered after ptxas (tools/sass_resched.py + the committed order)
RESCHED_VARIANT := 32, 8, 2, 2, 1, false, 1, 8, 1
RESCHED_ORDER   := $(PKG)/csrc/resched/pk_t32_r8_tj2_st2_cta_u1_mb8.order.json
RESCHED_INC     := $(PKG)/csrc/generated/force_resched_cubin.inc
$(RESCHED_INC): tools/sass_resched.py $(RESCHED_ORDER) $(PKG)/csrc/force_sm100.cuh $(PKG)/csrc/plan.hpp
	mkdir -p $(dir $@) build/resched && python3 tools/sass_resched.py "$(RESCHED_VARIANT)" build/resched/default.cubin --order-in $(RESCHED_ORDER) --emit-header $@

lib: $(LIB)
$(LIB): $(PKG)/csrc/context.cu $(PKG)/csrc/host_ic.cpp $(PKG)/csrc/force_sm100.cuh $(PKG)/csrc/field_sm100.cuh $(PKG)/csrc/neighbors_sm100.cuh $(PKG)/csrc/fof_sm100.cuh $(PKG)/csrc/phase_fof_sm100.cuh $(PKG)/csrc/groups_sm100.cuh $(PKG)/csrc/tracers_sm100.cuh $(PKG)/csrc/tidal_sm100.cuh $(PKG)/csrc/components_sm100.cuh $(PKG)/csrc/external_sm100.cuh $(PKG)/csrc/scf_sm100.cuh $(PKG)/csrc/integrate_sm100.cuh $(PKG)/csrc/plan.hpp include/b200nb.h $(RESCHED_INC)
	$(NVCC) $(NVFLAGS) -shared -o $@ $(PKG)/csrc/context.cu $(PKG)/csrc/host_ic.cpp -ldl

oracle: oracle/liboracle.so
oracle/liboracle.so: oracle/nbody_oracle.c oracle/nbody_oracle.h
	$(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ oracle/nbody_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ oracle/nbody_oracle.c -lm

# fp64 reference of the field / potential entry points (test infrastructure, beside the tests)
field_oracle: build/libfieldoracle.so
build/libfieldoracle.so: tests/field_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/field_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/field_oracle.c -lm)

# fp32 brute-force restatement of the nearest-neighbour definition (test infrastructure, beside the tests)
neighbors_oracle: build/libneighborsoracle.so
build/libneighborsoracle.so: tests/neighbors_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/neighbors_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/neighbors_oracle.c -lm)

# fp32 brute-force restatement of the friends-of-friends definition (test infrastructure, beside the tests)
fof_oracle: build/libfoforacle.so
build/libfoforacle.so: tests/fof_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O3 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/fof_oracle.c -lm || \
	$(ORACLE_CC) -O3 -ffp-contract=off -fPIC -shared -o $@ tests/fof_oracle.c -lm)

# fp32 brute-force restatement of the phase-space friends-of-friends definition (test infrastructure, beside the tests)
phase_fof_oracle: build/libphasefoforacle.so
build/libphasefoforacle.so: tests/phase_fof_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O3 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/phase_fof_oracle.c -lm || \
	$(ORACLE_CC) -O3 -ffp-contract=off -fPIC -shared -o $@ tests/phase_fof_oracle.c -lm)

# fp64 reference of the group potential and unbinding (test infrastructure, beside the tests)
groups_oracle: build/libgroupsoracle.so
build/libgroupsoracle.so: tests/groups_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/groups_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/groups_oracle.c -lm)

# the test-particle updates in the integrator's exact operation sequence, on the host (test infrastructure, beside the tests)
tracers_oracle: build/libtracersoracle.so
build/libtracersoracle.so: tests/tracers_oracle.c
	mkdir -p build && $(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/tracers_oracle.c -lm

# fp64 reference of the tidal tensor (test infrastructure, beside the tests)
tidal_oracle: build/libtidaloracle.so
build/libtidaloracle.so: tests/tidal_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/tidal_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/tidal_oracle.c -lm)

# fp64 reference of the field by component (test infrastructure, beside the tests)
components_oracle: build/libcomponentsoracle.so
build/libcomponentsoracle.so: tests/components_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/components_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/components_oracle.c -lm)

# the external-potential evaluator and the zero-self-gravity updates on the host (test infrastructure, beside the tests)
external_oracle: build/libexternaloracle.so
build/libexternaloracle.so: tests/external_oracle.c
	mkdir -p build && $(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/external_oracle.c -lm

# long-double restatement of the basis-function expansion (test infrastructure, beside the tests)
scf_oracle: build/libscforacle.so
build/libscforacle.so: tests/scf_oracle.c
	mkdir -p build && ($(ORACLE_CC) -O2 -ffp-contract=off -fopenmp -fPIC -shared -o $@ tests/scf_oracle.c -lm || \
	$(ORACLE_CC) -O2 -ffp-contract=off -fPIC -shared -o $@ tests/scf_oracle.c -lm)

# reference-side artefacts (need $(REF); outputs only under oracle/_ref/)
ref:
	bash oracle/build_ref.sh $(REF)

kbench: build/kbench
build/kbench: tools/kbench.cu $(PKG)/csrc/force_sm100.cuh $(PKG)/csrc/plan.hpp
	mkdir -p build && $(NVCC) $(ARCH) -O3 -std=c++17 -lineinfo -o $@ tools/kbench.cu -L/usr/local/cuda/lib64/stubs -lcuda

clean:
	rm -f $(LIB) oracle/liboracle.so build/kbench build/libfieldoracle.so build/libneighborsoracle.so build/libfoforacle.so build/libgroupsoracle.so build/libtracersoracle.so build/libtidaloracle.so build/libcomponentsoracle.so build/libexternaloracle.so build/libphasefoforacle.so build/libscforacle.so; rm -rf oracle/_ref

.PHONY: all lib oracle field_oracle neighbors_oracle fof_oracle groups_oracle tracers_oracle tidal_oracle components_oracle external_oracle phase_fof_oracle scf_oracle ref kbench clean
