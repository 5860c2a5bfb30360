# Builds libgdr_b200.so (the C-ABI library of include/gdr.h) for sm_100a, in-tree.
PKG      := graph-distillation-for-recommendation_b200
CSRC     := $(PKG)/csrc
OUT      := $(PKG)/lib/libgdr_b200.so
NVCC     ?= nvcc
NVFLAGS  := -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -lineinfo \
            -Xcompiler -fPIC,-fvisibility=hidden -Xptxas -v
SRCS     := $(wildcard $(CSRC)/*.cu)
OBJS     := $(patsubst $(CSRC)/%.cu,build/%.o,$(SRCS))

all: $(OUT)

build/%.o: $(CSRC)/%.cu $(CSRC)/common.cuh $(CSRC)/comm.cuh $(CSRC)/tc_common.cuh $(CSRC)/topk_common.cuh include/gdr.h
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; false)

$(OUT): $(OBJS)
	@mkdir -p $(PKG)/lib
	$(NVCC) -shared -o $@ $(OBJS) -lcuda -ldl

clean:
	rm -rf build $(OUT)
