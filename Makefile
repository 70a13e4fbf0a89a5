# stencil_b200 build: hand-written sm_100a CUDA, no cmake needed.
#   make            -> stencil_b200/libstencil_b200.so (C ABI + kernels) and lib/libstencil.a (C++ API, -rdc), plus
#                      bin/sb_mpirun, bin/jacobi3d_b200 and bin/test_exchange_multigpu (this repository's own drivers)
#   make drivers    -> bin/ : the REFERENCE's own drivers and Catch2 suites compiled, unchanged, from
#                      $(REF)/bin and $(REF)/test against OUR headers and library (needs $(REF))
#   make oracle     -> oracle/_build/liboracle.so (test infrastructure)
NVCC      ?= /usr/local/cuda/bin/nvcc
REF       ?= /root/reference
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -std=c++17 $(ARCH) -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Xcompiler -Wno-comment --expt-relaxed-constexpr
INC       := -Iinclude -Istencil_b200/csrc

# ---- core: kernels + C ABI (shared library, loaded by python and linked by the C++ API)
CSRC      := stencil_b200/csrc/box_copy.cu stencil_b200/csrc/jacobi.cu stencil_b200/csrc/astaroth.cu stencil_b200/csrc/reduce.cu \
             stencil_b200/csrc/capi.cu
COBJ      := $(patsubst stencil_b200/csrc/%.cu,build/csrc/%.o,$(CSRC))
SO        := stencil_b200/libstencil_b200.so

# ---- C++ API (static library with relocatable device code, like the reference's stencil::stencil)
APIDEFS   := -DSTENCIL_USE_MPI=1 -DSTENCIL_USE_CUDA=1 -DSTENCIL_USE_CUDA_AWARE_MPI=1 -DSTENCIL_USE_CUDA_GRAPH=1 \
             -DSTENCIL_SETUP_STATS=1 -DSTENCIL_OUTPUT_LEVEL=2 -DNDEBUG
APIINC    := -Iinclude -Iinclude/mpi_shim -I/usr/local/cuda/include/nvtx3
APIFLAGS  := -O3 -std=c++17 $(ARCH) -lineinfo -rdc=true --expt-extended-lambda -Xcompiler -fPIC -Xcompiler -Wall \
             -Xcompiler -Wno-comment -x cu $(APIDEFS) $(APIINC)
APISRC    := src/compat_kernels.cu src/local_domain.cu src/packer.cu src/translator.cu src/stencil.cu src/jacobi3d.cu \
             src/numeric.cpp src/timer.cpp src/rcstream.cpp src/topology.cpp src/gpu_topology.cpp \
             src/placement_intranoderandom.cpp
APIOBJ    := $(patsubst src/%,build/api/%.o,$(APISRC))
# the core objects are compiled a second time with -rdc for the static library
CAPIOBJ   := $(patsubst stencil_b200/csrc/%.cu,build/api/csrc_%.o,$(CSRC))
LIBA      := lib/libstencil.a
# the node-local MPI stand-in is a SEPARATE archive: link it only where no real MPI is (a second definition of MPI_*
# inside libstencil.a would shadow or clash with the real one)
LIBMPI    := lib/libmpi_shim.a

all: $(SO) $(LIBA) $(LIBMPI) bin/sb_mpirun bin/jacobi3d_b200 bin/test_exchange_multigpu

build/mpi_shim.o: src/mpi_shim.cpp include/mpi_shim/mpi.h
	@mkdir -p build
	g++ -O2 -std=c++17 -fPIC -Wall -Iinclude/mpi_shim -I/usr/local/cuda/include -c $< -o $@
$(LIBMPI): build/mpi_shim.o
	@mkdir -p lib
	rm -f $@ && ar rcs $@ $^

build/csrc/%.o: stencil_b200/csrc/%.cu $(wildcard stencil_b200/csrc/*.cuh) include/stencil_b200.h $(wildcard include/stencil/*.hpp)
	@mkdir -p $(dir $@)
	$(NVCC) $(NVCCFLAGS) $(INC) -c $< -o $@

build/numeric.o: src/numeric.cpp include/stencil/numeric.hpp
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) $(INC) -c $< -o $@

$(SO): $(COBJ) build/numeric.o
	$(NVCC) $(ARCH) -shared -o $@ $^ -cudart shared

build/api/%.o: src/% $(wildcard include/stencil/*) include/stencil_b200.h include/mpi_shim/mpi.h
	@mkdir -p $(dir $@)
	$(NVCC) $(APIFLAGS) -c $< -o $@

build/api/csrc_%.o: stencil_b200/csrc/%.cu $(wildcard stencil_b200/csrc/*.cuh) include/stencil_b200.h $(wildcard include/stencil/*.hpp)
	@mkdir -p $(dir $@)
	$(NVCC) $(APIFLAGS) -Istencil_b200/csrc -c $< -o $@

$(LIBA): $(APIOBJ) $(CAPIOBJ)
	@mkdir -p lib
	rm -f $@ && ar rcs $@ $^

# ---- the reference's unchanged drivers / tests against our library
DRVFLAGS  := -O3 -std=c++14 $(ARCH) -lineinfo -rdc=true --expt-extended-lambda -Xcompiler -w -w -x cu $(APIDEFS) \
             -DCATCH_CONFIG_NO_POSIX_SIGNALS $(APIINC) -I$(REF)/thirdparty -I$(REF)/bin
DRVLINK    = $(ARCH) -rdc=true -L/usr/local/cuda/lib64/stubs -lnvidia-ml -ldl -lcudart -lrt
# this repository's own drivers and checks: built by `make` without $(REF)
OWNFLAGS  := $(filter-out -I$(REF)/thirdparty -I$(REF)/bin,$(DRVFLAGS))
DRIVERS   := jacobi3d jacobi3d_strong bench_exchange bench_pack exchange_weak exchange_strong
TESTCUDA  := test_cuda_main test_cuda_align test_cuda_local_domain test_cuda_pack test_cuda_packer test_cuda_rcstream \
             test_cuda_translate test_cuda_translate_kernel test_cuda_gpu_topo test_exchange
TESTCPU   := test_cpu_main test_cpu_partition test_cpu_numeric test_cpu_radius test_cpu_accessor test_cpu_tx \
             test_cpu_mat2d test_cpu_qap

build/drv/%.o: $(REF)/bin/%.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(DRVFLAGS) -c $< -o $@
build/drv/statistics.o: $(REF)/bin/statistics.cpp
	@mkdir -p $(dir $@)
	$(NVCC) $(DRVFLAGS) -c $< -o $@
build/drv/t_%.o: $(REF)/test/%.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(DRVFLAGS) -c $< -o $@
build/drv/t_%.o: $(REF)/test/%.cpp $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(DRVFLAGS) -c $< -o $@

bin/%: build/drv/%.o build/drv/statistics.o $(LIBA) $(LIBMPI)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $< build/drv/statistics.o $(LIBA) $(LIBMPI)
bin/test_cuda: $(patsubst %,build/drv/t_%.o,$(TESTCUDA)) $(LIBA)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $(patsubst %,build/drv/t_%.o,$(TESTCUDA)) $(LIBA) $(LIBMPI)
bin/test_cpu: $(patsubst %,build/drv/t_%.o,$(TESTCPU)) $(LIBA)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $(patsubst %,build/drv/t_%.o,$(TESTCPU)) $(LIBA) $(LIBMPI)

# our own driver: the reference's jacobi3d loop over stencil::FusedJacobi3d (no reference sources involved)
build/drv/jacobi3d_b200.o: drivers/jacobi3d_b200.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(OWNFLAGS) -c $< -o $@
bin/jacobi3d_b200: build/drv/jacobi3d_b200.o $(LIBA)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $< $(LIBA) $(LIBMPI)

# launcher of the node-local MPI shim (one rank per GPU without an MPI installation)
bin/sb_mpirun: drivers/sb_mpirun.cpp $(LIBMPI)
	@mkdir -p bin
	g++ -O2 -std=c++17 -o $@ $< $(LIBMPI) -L/usr/local/cuda/lib64 -lcudart -lrt -lpthread

# the baseline exchange driver (oracle/ref/ref_exchange_uniform.cu) against OUR library
build/drv/exchange_uniform.o: oracle/ref/ref_exchange_uniform.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(DRVFLAGS) -c $< -o $@

# our own multi-GPU check of the C++ API
build/drv/test_exchange_multigpu.o: tests/cpp/test_exchange_multigpu.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(OWNFLAGS) -c $< -o $@
bin/test_exchange_multigpu: build/drv/test_exchange_multigpu.o $(LIBA) $(LIBMPI)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $< $(LIBA) $(LIBMPI)

# the reference's astaroth driver (its own MHD kernels; halos through our library), unchanged
ASTRO     := astaroth kernels astaroth_utils
ASTROFLAGS := $(filter-out -I$(REF)/bin,$(DRVFLAGS)) --use_fast_math -I$(REF)/astaroth -DAC_DEFAULT_CONFIG=\"oracle/_ref/astaroth.conf\"
build/drv/astro_%.o: $(REF)/astaroth/%.cu $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(ASTROFLAGS) -c $< -o $@
build/drv/astro_statistics.o: $(REF)/astaroth/statistics.cpp
	@mkdir -p $(dir $@)
	$(NVCC) $(ASTROFLAGS) -c $< -o $@
bin/astaroth: $(patsubst %,build/drv/astro_%.o,$(ASTRO)) build/drv/astro_statistics.o $(LIBA)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ $(patsubst %,build/drv/astro_%.o,$(ASTRO)) build/drv/astro_statistics.o $(LIBA) $(LIBMPI)

# the same driver with the reference's kernels.cu REPLACED by ours (src/astaroth_kernels.cu -> sb_astaroth_substep)
build/drv/astro_b200_kernels.o: src/astaroth_kernels.cu include/stencil_b200.h $(wildcard include/stencil/*)
	@mkdir -p $(dir $@)
	$(NVCC) $(ASTROFLAGS) -Iinclude -c $< -o $@
bin/astaroth_b200: build/drv/astro_astaroth.o build/drv/astro_astaroth_utils.o build/drv/astro_b200_kernels.o build/drv/astro_statistics.o $(LIBA)
	@mkdir -p bin
	$(NVCC) $(DRVLINK) -o $@ build/drv/astro_astaroth.o build/drv/astro_astaroth_utils.o build/drv/astro_b200_kernels.o build/drv/astro_statistics.o $(LIBA) $(LIBMPI)

drivers: bin/sb_mpirun bin/jacobi3d_b200 $(patsubst %,bin/%,$(DRIVERS)) bin/test_cuda bin/test_cpu bin/exchange_uniform bin/astaroth bin/astaroth_b200 bin/test_exchange_multigpu

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf build $(SO) lib bin

.PHONY: all drivers oracle clean
.SECONDARY:
