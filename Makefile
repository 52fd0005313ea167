# Builds librt_b200.so (sm_100a only) in-tree, the oracle, and the apps.
NVCC      ?= /usr/local/cuda/bin/nvcc
CXX       ?= g++
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := $(ARCH) -std=c++17 -O3 -lineinfo -Xcompiler -fPIC -Xcompiler -Wall -Xptxas -v --expt-relaxed-constexpr
CXXFLAGS  := -std=c++17 -O2 -fPIC -Wall -Wextra
PKG       := raytracing_renderer_cuda_b200
CSRC      := $(PKG)/csrc
OBJDIR    := build
LIB       := $(PKG)/librt_b200.so

CU_SRCS   := $(CSRC)/rt_api.cu $(CSRC)/rt_kernels.cu $(CSRC)/rt_wavefront.cu $(CSRC)/rt_lbvh.cu $(CSRC)/rt_jpeg.cu $(CSRC)/rt_jpeg_decode.cu $(CSRC)/rt_multi.cu $(CSRC)/rt_denoise.cu $(CSRC)/rt_adaptive.cu $(CSRC)/rt_selftest.cu
CPP_SRCS  := $(CSRC)/rt_host.cpp $(CSRC)/rt_bvh_host.cpp $(CSRC)/rt_jpeg_decode_host.cpp
CU_OBJS   := $(patsubst $(CSRC)/%.cu,$(OBJDIR)/%.o,$(CU_SRCS))
CPP_OBJS  := $(patsubst $(CSRC)/%.cpp,$(OBJDIR)/%.o,$(CPP_SRCS))
HDRS      := $(wildcard $(CSRC)/*.cuh $(CSRC)/*.hpp include/*.h include/rt/*.hpp)

all: $(LIB) oracle apps

lib: $(LIB)

$(OBJDIR)/%.o: $(CSRC)/%.cu $(HDRS)
	@mkdir -p $(OBJDIR)
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> $(OBJDIR)/$*.ptxas.log || (cat $(OBJDIR)/$*.ptxas.log; false)

$(OBJDIR)/%.o: $(CSRC)/%.cpp $(HDRS)
	@mkdir -p $(OBJDIR)
	$(CXX) $(CXXFLAGS) -c $< -o $@

$(LIB): $(CU_OBJS) $(CPP_OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $^ -lcudart

oracle:
	$(MAKE) -C oracle

apps: $(LIB)
	$(MAKE) -C apps

clean:
	rm -rf $(OBJDIR) $(LIB)
	$(MAKE) -C oracle clean || true
	$(MAKE) -C apps clean || true

.PHONY: all lib oracle apps clean
