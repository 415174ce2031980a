# Builds libctr_b200.so (sm_100a only) in-tree; `python -c "import __graft_entry__ as g; g.build()"` calls this.
CUDA_HOME ?= /usr/local/cuda
# nvcc from PATH, else from the CUDA install (a plain user's PATH often lacks $(CUDA_HOME)/bin)
NVCC      ?= $(if $(shell command -v nvcc),nvcc,$(CUDA_HOME)/bin/nvcc)
ARCH      := -gencode arch=compute_100a,code=sm_100a
NVCCFLAGS := -O3 -std=c++17 -lineinfo $(ARCH) -Xcompiler -fPIC,-Wall,-Wno-unused-function -Xptxas -v
SRC_DIR   := tf_repos_b200/csrc
SRCS      := $(wildcard $(SRC_DIR)/*.cu)
OBJS      := $(patsubst $(SRC_DIR)/%.cu,build/%.o,$(SRCS))
LIB       := tf_repos_b200/libctr_b200.so

all: $(LIB)

build/%.o: $(SRC_DIR)/%.cu $(wildcard $(SRC_DIR)/*.cuh) include/ctr_b200.h
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -c $< -o $@ 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	$(NVCC) $(ARCH) -shared -o $@ $(OBJS) -cudart static

clean:
	rm -rf build $(LIB)
.PHONY: all clean
