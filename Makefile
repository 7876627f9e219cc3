# Builds the product library (CUDA, sm_100a only) and the test-only artefacts.
#   make lib       -> libgoldilocks_b200/libgoldilocks_b200.so   (the C ABI of include/goldilocks_b200.h)
#   make hostsim   -> tests/hostsim/_hostsim.so                  (device math compiled for the host; tests only)
#   make oracle    -> oracle/liboracle.so (+ oracle/_ref/*.so with REF=<libgoldilocks source tree>; tests/bench baseline only)
NVCC      ?= nvcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -O3 -lineinfo -std=c++17 -Xcompiler -fPIC,-fvisibility=hidden $(EXTRA_NVCCFLAGS)
CSRC      := libgoldilocks_b200/csrc
OBJDIR    ?= build/obj
KERNELS   := $(wildcard $(CSRC)/k_*.cu)
OBJS      := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(KERNELS)) $(OBJDIR)/abi.o
HDRS      := $(wildcard $(CSRC)/*.cuh) $(wildcard $(CSRC)/*.h) include/goldilocks_b200.h
LIB       ?= libgoldilocks_b200/libgoldilocks_b200.so

.PHONY: all lib hostsim oracle tools clean
all: lib hostsim oracle tools
tools: tools/imad_peak tools/single_calls
tools/imad_peak: tools/imad_peak.cu
	$(NVCC) $(ARCH) -O3 -lineinfo -o $@ $<
tools/single_calls: tools/single_calls.cpp $(LIB) include/goldilocks_b200.h
	$(CXX) -O2 -std=c++17 -pthread -Iinclude -o $@ $< -Llibgoldilocks_b200 -lgoldilocks_b200 -Wl,-rpath,'$$ORIGIN/../libgoldilocks_b200'
lib: $(LIB)

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS_$*) $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) -Xptxas -v -c -o $@ $< 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; false)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -cudart static -o $@ $(OBJS)

hostsim: tests/hostsim/_hostsim.so
tests/hostsim/_hostsim.so: tests/hostsim/hostsim.cpp $(HDRS)
	$(CXX) -std=c++17 -O2 -fPIC -shared -DGF_CHECK_BOUNDS -DGF_COUNT_OPS -o $@ $< -lpthread

oracle:
	$(MAKE) -C oracle all

clean:
	rm -rf build $(LIB) tests/hostsim/_hostsim.so
	$(MAKE) -C oracle clean
