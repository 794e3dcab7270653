# Builds the product libraries in-tree (they travel to the GPU box with the
# snapshot):
#   form_b200/lib/libformgpu.so   CUDA hot path + C-ABI (include/formgpu.h)
#   form_b200/lib/libformhost.so  C++ host facade (form::Estimator, batch replay)
#   form_b200/lib/libformsynth.so synthetic scans + SE(3) hooks only: no CUDA dependency, so that the
#                                 CPU baseline / oracle tests never map the product's CUDA library
# and, for tests / bench baselines only, oracle/_build/liboracle.so and oracle/_ref/libformref.so.
NVCC      ?= /usr/local/cuda/bin/nvcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVFLAGS   := $(ARCH) -O3 -std=c++17 -lineinfo -Xcompiler -fPIC -Iinclude -Iform_b200/csrc
# index-determining kernels: no FMA contraction so results match the oracle bit for bit
EXACT     := -fmad=false
CXXFLAGS  := -O3 -std=c++17 -fPIC -pthread -ffp-contract=off -Wall -Iinclude -Iform_b200/host
LIBDIR    := form_b200/lib
OBJDIR    := build/obj

GPU_OBJS  := $(OBJDIR)/extract.o $(OBJDIR)/map_assoc.o $(OBJDIR)/linearize.o $(OBJDIR)/moments.o $(OBJDIR)/api.o $(OBJDIR)/api_stage2.o $(OBJDIR)/api_stage3.o $(OBJDIR)/api_batch.o $(OBJDIR)/comm.o $(OBJDIR)/organize.o $(OBJDIR)/api_cloud.o
HOST_SRCS := $(wildcard form_b200/host/src/*.cpp)
HOST_OBJS := $(HOST_SRCS:form_b200/host/src/%.cpp=$(OBJDIR)/host_%.o)
CSRC_HDRS := $(wildcard form_b200/csrc/*.hpp) $(wildcard form_b200/csrc/*.cuh) include/formgpu.h
HOST_HDRS := $(wildcard form_b200/host/form/*.hpp) include/formgpu.h

PYTHON    ?= python3
PYEXT     := python/form/_core$(shell $(PYTHON) -c "import sysconfig; print(sysconfig.get_config_var('EXT_SUFFIX'))")

all: $(LIBDIR)/libformgpu.so $(LIBDIR)/libformhost.so $(LIBDIR)/libformsynth.so $(PYEXT) oracle

# form._core: the reference's Python surface (python/bindings.cpp) with pybind11
$(PYEXT): python/bindings.cpp $(HOST_HDRS) $(LIBDIR)/libformgpu.so
	$(CXX) -O2 -std=c++17 -fPIC -shared -pthread -ffp-contract=off -fvisibility=hidden -Iinclude -Iform_b200/host \
	    $(shell $(PYTHON) -m pybind11 --includes) $< -o $@ -L$(LIBDIR) -lformgpu -Wl,-rpath,'$$ORIGIN/../../form_b200/lib'

$(OBJDIR)/extract.o: form_b200/csrc/extract.cu $(CSRC_HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXACT) -Xptxas -v -c $< -o $@

$(OBJDIR)/map_assoc.o: form_b200/csrc/map_assoc.cu $(CSRC_HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXACT) -Xptxas -v -c $< -o $@

$(OBJDIR)/organize.o: form_b200/csrc/organize.cu $(CSRC_HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) $(EXACT) -Xptxas -v -c $< -o $@

$(OBJDIR)/%.o: form_b200/csrc/%.cu $(CSRC_HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@

$(LIBDIR)/libformgpu.so: $(GPU_OBJS)
	@mkdir -p $(LIBDIR)
	$(NVCC) $(ARCH) -shared -o $@ $(GPU_OBJS) -cudart static -ldl

$(OBJDIR)/host_%.o: form_b200/host/src/%.cpp $(HOST_HDRS)
	@mkdir -p $(OBJDIR)
	$(CXX) $(CXXFLAGS) -c $< -o $@

$(LIBDIR)/libformhost.so: $(HOST_OBJS) $(LIBDIR)/libformgpu.so
	$(CXX) -shared -pthread -o $@ $(HOST_OBJS) -L$(LIBDIR) -lformgpu -Wl,-rpath,'$$ORIGIN'

$(LIBDIR)/libformsynth.so: $(OBJDIR)/host_synth_capi.o
	@mkdir -p $(LIBDIR)
	$(CXX) -shared -pthread -Wl,--no-undefined -Wl,-Bsymbolic -o $@ $<

# oracle/_ref: FORM's own stage-1/2 sources compiled from /root/reference against API
# stand-ins (test infrastructure; skipped where the reference tree is absent)
oracle: $(LIBDIR)/libformgpu.so
	$(MAKE) -s -C oracle
	$(MAKE) -s -C oracle/ref

clean:
	rm -rf build $(LIBDIR)/*.so oracle/_build oracle/_ref python/form/_core*.so

.PHONY: all oracle clean
