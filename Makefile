# Builds the three native artefacts, all in-tree (the .so files travel to the GPU box with gpurun):
#   pathtracer_rs_b200/lib/libptrs_b200.so   the product: sm_100a kernels + C ABI (include/ptrs_b200.h)
#   pathtracer_rs_b200/lib/libptrs_host.so   host-side scene preparation (BVH build, importers' work)
#   oracle/_build/liboracle.so               CPU oracle (test infrastructure)
# -fmad=false / -ffp-contract=off everywhere: the reference (rustc) never fuses multiply-add, and
# bit-exact hit parity depends on it.
NVCC      ?= /usr/local/cuda/bin/nvcc
HOSTCXX   := /usr/bin/g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCBASE  := -std=c++17 -O3 $(ARCH) -lineinfo -ftz=false -ccbin $(HOSTCXX) -Xcompiler -fPIC -diag-suppress 177 -Xptxas -v
# exact units: Sobol, camera rays, BVH traversal, triangle test — bit-identical to the CPU path
NVCCFLAGS := $(NVCCBASE) -fmad=false -prec-div=true -prec-sqrt=true
# shading units: everything downstream of sin/cos/exp is toleranced anyway (DESIGN.md §3), so FMA
# contraction and the 2-ulp division / square root are allowed there
SHADEFLAGS := $(NVCCBASE) -fmad=true -prec-div=false -prec-sqrt=false
CXXFLAGS  := -std=c++17 -O2 -ffp-contract=off -fno-fast-math -fopenmp -fPIC -Wall -Wno-unused-function

CS   := pathtracer_rs_b200/csrc
HS   := pathtracer_rs_b200/host
LIB  := pathtracer_rs_b200/lib
OBJ  := build/obj
BLOB := $(abspath pathtracer_rs_b200/data/sobol_tables.bin)

DEV_HDRS  := $(wildcard $(CS)/*.cuh) $(CS)/launch.hpp $(CS)/handles.hpp include/ptrs_b200.h
SHADE_OBJ := $(foreach m,0 1 2 3 4 5,$(OBJ)/k_shade_$(m).o $(OBJ)/k_shade_exact_$(m).o)
CUDA_OBJ  := $(OBJ)/ptrs_b200.o $(OBJ)/multi_gpu.o $(OBJ)/k_probe_fast.o $(OBJ)/k_probe_exact.o $(OBJ)/k_trace.o $(OBJ)/k_misc.o $(OBJ)/k_bvh.o $(OBJ)/k_sah.o $(OBJ)/k_tables.o $(SHADE_OBJ) $(OBJ)/sobol_blob.o

all: $(LIB)/libptrs_b200.so $(LIB)/libptrs_host.so oracle/_build/liboracle.so examples

examples: $(LIB)/libptrs_b200.so $(LIB)/libptrs_host.so
	$(MAKE) -C examples

$(OBJ)/%.o: $(CS)/%.cu $(DEV_HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ > $(OBJ)/$*.ptxas.log 2>&1 || (cat $(OBJ)/$*.ptxas.log; false)

$(OBJ)/k_probe_fast.o: $(CS)/k_probe.cu $(DEV_HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(SHADEFLAGS) -DPT_PROBE_EXACT=0 -c $< -o $@ > $(OBJ)/k_probe_fast.ptxas.log 2>&1 || (cat $(OBJ)/k_probe_fast.ptxas.log; false)
$(OBJ)/k_probe_exact.o: $(CS)/k_probe.cu $(DEV_HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -DPT_PROBE_EXACT=1 -c $< -o $@ > $(OBJ)/k_probe_exact.ptxas.log 2>&1 || (cat $(OBJ)/k_probe_exact.ptxas.log; false)

# parity mode (PTRS_RENDER_EXACT_SHADING): the same shade kernels with the exact units' arithmetic
$(OBJ)/k_shade_exact_%.o: $(CS)/k_shade.cu $(DEV_HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(NVCCFLAGS) -DPT_SHADE_EXACT=1 -DPT_SHADE_MAT=$* -c $< -o $@ > $(OBJ)/k_shade_exact_$*.ptxas.log 2>&1 || (cat $(OBJ)/k_shade_exact_$*.ptxas.log; false)

$(OBJ)/k_shade_%.o: $(CS)/k_shade.cu $(DEV_HDRS)
	@mkdir -p $(OBJ)
	$(NVCC) $(SHADEFLAGS) -DPT_SHADE_MAT=$* -c $< -o $@ > $(OBJ)/k_shade_$*.ptxas.log 2>&1 || (cat $(OBJ)/k_shade_$*.ptxas.log; false)

$(OBJ)/sobol_blob.o: $(CS)/sobol_blob.S $(BLOB)
	@mkdir -p $(OBJ)
	$(HOSTCXX) -c -DSOBOL_BLOB_PATH='"$(BLOB)"' $< -o $@

$(LIB)/libptrs_b200.so: $(CUDA_OBJ)
	@mkdir -p $(LIB)
	$(NVCC) $(ARCH) -ccbin $(HOSTCXX) -shared -o $@ $(CUDA_OBJ) -cudart static -ldl -lpthread

$(LIB)/libptrs_host.so: $(wildcard $(HS)/*.cpp) $(wildcard $(HS)/*.hpp) include/ptrs_b200.h
	@mkdir -p $(LIB)
	$(HOSTCXX) $(CXXFLAGS) -shared $(wildcard $(HS)/*.cpp) -o $@ -lz

oracle/_build/liboracle.so: oracle/oracle_capi.cpp $(wildcard oracle/*.hpp) include/ptrs_b200.h
	$(MAKE) -C oracle

clean:
	rm -rf build $(LIB) oracle/_build

.PHONY: all clean examples
