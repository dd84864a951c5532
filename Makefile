# Builds the C-ABI library of hand-written sm_100a kernels (cross-compiles without a GPU).
NVCC      ?= /usr/local/cuda/bin/nvcc
PKG       := smb-vision_b200
CSRC      := $(PKG)/csrc
LIB       := $(PKG)/lib/libsmbv_b200.so
SRCS      := $(wildcard $(CSRC)/*.cu)
OBJS      := $(patsubst $(CSRC)/%.cu,build/%.o,$(SRCS))
NVCCFLAGS := -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -Xcompiler -fPIC \
             -Xptxas -v --expt-relaxed-constexpr -Iinclude

all: $(LIB)

build/%.o: $(CSRC)/%.cu $(CSRC)/common.cuh include/smbv_b200.h
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; false)

$(LIB): $(OBJS)
	@mkdir -p $(PKG)/lib
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -o $@ $(OBJS) -cudart static

clean:
	rm -rf build $(LIB)
.PHONY: all clean
