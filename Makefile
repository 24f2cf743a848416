# Builds libcoverage_cuda.so (sm_100a) and the CPU oracle (test infrastructure).
EXTRA     ?=
NVCC      ?= /usr/local/cuda/bin/nvcc
GCC       ?= /usr/bin/gcc
PKG       := maximumareacoverageoptimization.jl_b200
CSRC      := $(PKG)/csrc
LIB       := $(PKG)/libcoverage_cuda.so
ORACLE    := oracle/libcoverage_oracle.so
NVCCFLAGS := --threads 0 -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo --fmad=false \
             -Xcompiler -fPIC,-O2,-fno-fast-math,-ffp-contract=off,-fvisibility=hidden,-pthread -Xptxas -v $(EXTRA)
SRCS      := $(CSRC)/cov_api.cu $(CSRC)/cov_kernels.cu $(CSRC)/cov_span_small.cu $(CSRC)/cov_span_cta.cu $(CSRC)/cov_grid_kernels.cu $(CSRC)/cov_mads.cu \
             $(CSRC)/cov_region.cu $(CSRC)/cov_horizon.cu
HDRS      := $(wildcard $(CSRC)/*.h $(CSRC)/*.cuh) include/coverage_cuda.h

all: $(LIB) $(ORACLE)

$(LIB): $(SRCS) $(HDRS)
	$(NVCC) $(NVCCFLAGS) -shared -o $@ $(SRCS) -cudart static

$(ORACLE): oracle/coverage_oracle.c
	$(GCC) -O2 -fPIC -shared -pthread -ffp-contract=off -fno-fast-math -fvisibility=hidden -o $@ $< -lm

# checking variant: device asserts on every framebuffer / plane index (compute-sanitizer is closed on the pool)
debug-bounds:
	mkdir -p build/variants
	$(NVCC) $(filter-out -Xptxas -v,$(NVCCFLAGS)) -DCOV_DEBUG_BOUNDS -shared -o build/variants/lib_debug_bounds.so $(SRCS) -cudart static
	@echo 'run: COVERAGE_CUDA_LIB=$$PWD/build/variants/lib_debug_bounds.so python -m pytest tests -m gpu'

# checking variant: the paint-then-sweep mode paints whole words with atomicOr instead of plain stores (DESIGN.md 2.4)
strict-atomics:
	mkdir -p build/variants
	$(NVCC) $(filter-out -Xptxas -v,$(NVCCFLAGS)) -DCOV_STRICT_ATOMICS -shared -o build/variants/lib_strict_atomics.so $(SRCS) -cudart static
	@echo 'run: COVERAGE_CUDA_LIB=$$PWD/build/variants/lib_strict_atomics.so python -m pytest tests -m gpu'

clean:
	rm -f $(LIB) $(ORACLE)
.PHONY: all clean debug-bounds strict-atomics
