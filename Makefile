# ptb200 — build everything that travels to the GPU box.
#   make            -> raytracing-rust_b200/libptb200.so (CUDA, sm_100a) + oracle/liboracle.so (test infrastructure)
#   make cli        -> raytracing-rust_b200/ptb200-cli (C++ frontend mirroring src/parameters.rs + `--backend cuda`)
PKG      := raytracing-rust_b200
NVCC     ?= nvcc
# -fmad=false: the reference (rustc) never contracts a*b+c; hit/miss decisions must match the oracle bit for bit.
NVFLAGS  ?= -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -fmad=false \
            -Xcompiler -fPIC,-Wall,-Wextra,-Wno-unused-parameter -Xptxas -v
CU_SRCS  := $(PKG)/csrc/context.cu $(PKG)/csrc/lbvh_build.cu $(PKG)/csrc/cwbvh_build.cu $(PKG)/csrc/sah_build.cu $(PKG)/csrc/wavefront.cu $(PKG)/csrc/multi.cu $(PKG)/csrc/denoise.cu
CPP_SRCS := $(PKG)/host/ssml_loader.cpp $(PKG)/host/image_out.cpp $(PKG)/host/image_in.cpp
HDRS     := include/ptb200.h $(wildcard $(PKG)/csrc/*.cuh) $(wildcard $(PKG)/csrc/*.h)
OBJS     := $(CU_SRCS:.cu=.o) $(CPP_SRCS:.cpp=.o)

all: $(PKG)/libptb200.so cli oracle

$(PKG)/csrc/%.o: $(PKG)/csrc/%.cu $(HDRS)
	$(NVCC) $(NVFLAGS) -c $< -o $@ 2> $@.ptxas.log || (cat $@.ptxas.log; false)
$(PKG)/host/%.o: $(PKG)/host/%.cpp include/ptb200.h
	$(CXX) -O2 -std=c++17 -fPIC -Wall -Wextra -fno-fast-math -ffp-contract=off -c $< -o $@

$(PKG)/libptb200.so: $(OBJS)
	$(NVCC) -shared -gencode arch=compute_100a,code=sm_100a -o $@ $(OBJS) -cudart static -ldl

cli: $(PKG)/ptb200-cli
$(PKG)/ptb200-cli: $(PKG)/host/cli_main.cpp $(PKG)/libptb200.so include/ptb200.h
	$(CXX) -O2 -std=c++17 -Wall -Wextra -o $@ $(PKG)/host/cli_main.cpp -L$(PKG) -lptb200 -Wl,-rpath,'$$ORIGIN' -ldl -lpthread

oracle: oracle/libvisibility_oracle.so oracle/librefit_oracle.so oracle/libaov_oracle.so oracle/libdenoise_oracle.so \
        oracle/libmotion_oracle.so oracle/libtemporal_oracle.so
	$(MAKE) -C oracle
# test infrastructure beside liboracle.so: the reference's visibility queries for a batch (oracle/visibility_api.cpp)
oracle/libvisibility_oracle.so: oracle/visibility_api.cpp $(wildcard oracle/*.hpp) include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<
# ... and the refit of a kept binary tree (oracle/refit_api.cpp, PTB_BUILD_REFIT)
oracle/librefit_oracle.so: oracle/refit_api.cpp $(wildcard oracle/*.hpp) include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<
# ... and the denoiser feature buffers of the render's camera rays (oracle/aov_api.cpp, ptb_render_aov)
oracle/libaov_oracle.so: oracle/aov_api.cpp $(wildcard oracle/*.hpp) include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<
# ... and the denoiser over the beauty and AOV sums (oracle/denoise_api.cpp, ptb_denoise)
oracle/libdenoise_oracle.so: oracle/denoise_api.cpp include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<
# ... and the motion vectors of ptb_render_aov after a mark (oracle/motion_api.cpp, over the AOV oracle's scene)
oracle/libmotion_oracle.so: oracle/motion_api.cpp oracle/aov_api.cpp $(wildcard oracle/*.hpp) include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<
# ... and one step of the temporal denoiser (oracle/temporal_api.cpp, over the spatial oracle's helpers)
oracle/libtemporal_oracle.so: oracle/temporal_api.cpp oracle/denoise_api.cpp include/ptb200.h
	$(CXX) -O2 -std=c++17 -fno-fast-math -ffp-contract=off -fPIC -Wall -Wextra -pthread -shared -o $@ $<

clean:
	rm -f $(OBJS) $(PKG)/csrc/*.ptxas.log $(PKG)/libptb200.so $(PKG)/ptb200-cli oracle/libvisibility_oracle.so oracle/librefit_oracle.so oracle/libaov_oracle.so oracle/libdenoise_oracle.so \
	      oracle/libmotion_oracle.so oracle/libtemporal_oracle.so
	$(MAKE) -C oracle clean
.PHONY: all oracle clean cli
