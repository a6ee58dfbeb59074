# Builds the CUDA library (sm_100a only), the CLI and the CPU oracle (test infrastructure).
NVCC ?= nvcc
ARCH := -gencode arch=compute_100a,code=sm_100a
NVFLAGS := $(ARCH) -std=c++17 -O3 -lineinfo -Xcompiler -fPIC,-Wall,-Wextra -Xptxas -v
SRC := rttnw_b200/csrc
LIB := rttnw_b200/lib/librttnw_b200.so
CLI := rttnw_b200/lib/rttnw
HDRS := include/rttnw_b200.h $(SRC)/device_types.h $(SRC)/flatten.hpp $(SRC)/kernels.cuh $(SRC)/shade2.cuh $(SRC)/shade2_body.cuh $(SRC)/aov_body.cuh $(SRC)/order.cuh $(SRC)/trace2.cuh $(SRC)/trace3.cuh $(SRC)/lbvh.cuh $(SRC)/sah_build.cuh $(SRC)/adaptive.cuh $(SRC)/aov.cuh $(SRC)/denoise.cuh $(SRC)/scene_api.hpp

all: $(LIB) $(CLI) oracle

$(LIB): $(SRC)/api.cu $(SRC)/flatten.cpp $(SRC)/scenes.cpp $(SRC)/png_io.cpp $(HDRS)
	@mkdir -p rttnw_b200/lib
	$(NVCC) $(NVFLAGS) -shared -o $@ $(SRC)/api.cu $(SRC)/flatten.cpp $(SRC)/scenes.cpp $(SRC)/png_io.cpp -lz -ldl

$(CLI): $(SRC)/cli.cpp $(LIB) include/rttnw_b200.h
	g++ -std=c++17 -O2 -Wall -Wextra -o $@ $(SRC)/cli.cpp -Iinclude -Lrttnw_b200/lib -lrttnw_b200 -lpthread -Wl,-rpath,'$$ORIGIN'

oracle:
	$(MAKE) -C oracle

clean:
	rm -rf rttnw_b200/lib oracle/_build
.PHONY: all oracle clean
