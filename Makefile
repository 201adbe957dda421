# Builds libraytracing_cuda.so (the product) for sm_100a, the CPU oracle and the CPU kernel-body harness.
NVCC ?= nvcc
PKG := opencl-raytracing_b200
CSRC := $(PKG)/csrc
NVCCFLAGS := -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -std=c++17 -Xcompiler -fPIC -Xcompiler -fvisibility=hidden $(NVCCFLAGS_EXTRA)
HDRS := $(wildcard $(CSRC)/*.h) $(CSRC)/kernels.cuh include/rtcuda.h

all: $(PKG)/libraytracing_cuda.so oracle/liboracle.so tests/hostsim/libhostsim.so tests/hostsim/libhostsim_update.so \
	tests/hostsim/libhostsim_query.so tests/hostsim/liboracle_query.so tests/hostsim/libhostsim_radiance.so tests/hostsim/liboracle_radiance.so \
	tests/hostsim/libhostsim_surfaces.so tests/hostsim/liboracle_surfaces.so oracle_ref

# the reference's own C++ device headers compiled for the host (checker of the oracle; no-op when /root/reference is absent)
.PHONY: oracle_ref
oracle_ref:
	$(MAKE) -C oracle/ref_shim

# wavefront kernels: FMA contraction on, 2-ulp division / sqrt (the beauty plane is gated statistically; the
# strict-tolerance AOV kernels live in kernels_aov.cu and keep IEEE division, sqrt and unfused multiply-add)
# RT_FAST_RCP: 1 / direction of the slab tests is a bare MUFU.RCP (rt_traverse.h safe_rcp_dir; only the conservative box
# culling reads it): k_extend 61.4 -> 60.6 ms, k_shadow 112.9 -> 110.7 ms on C3 (profiles/r4p_ab.log)
FASTDIV ?= -prec-div=false -prec-sqrt=false -DRT_FAST_RCP=1
build/kernels.o: $(CSRC)/kernels.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) $(FASTDIV) -c $< -o $@

build/kernels_aov.o: $(CSRC)/kernels_aov.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -fmad=false -c $< -o $@

build/api.o: $(CSRC)/api.cu $(HDRS)
	@mkdir -p build
	$(NVCC) $(NVCCFLAGS) -c $< -o $@

$(PKG)/libraytracing_cuda.so: build/kernels.o build/kernels_aov.o build/api.o
	$(NVCC) -shared -o $@ $^ -lcudart_static -lrt -lpthread -ldl

oracle/liboracle.so: oracle/oracle.cpp include/rtcuda.h
	$(MAKE) -C oracle liboracle.so

tests/hostsim/libhostsim.so: tests/hostsim/hostsim.cpp $(HDRS)
	g++ -O2 -std=c++17 -fPIC -shared -pthread -o $@ $<

# the scene-update refit on the CPU (includes hostsim.cpp)
tests/hostsim/libhostsim_update.so: tests/hostsim/hostsim_update.cpp tests/hostsim/hostsim.cpp $(HDRS)
	g++ -O2 -std=c++17 -fPIC -shared -pthread -o $@ $<

# the ray queries on the CPU (includes hostsim.cpp)
tests/hostsim/libhostsim_query.so: tests/hostsim/hostsim_query.cpp tests/hostsim/hostsim.cpp $(HDRS)
	g++ -O2 -std=c++17 -fPIC -shared -pthread -o $@ $<

# their reference: the oracle's traverse_bvh per caller-supplied ray (includes oracle/oracle.cpp, built with the oracle's flags)
tests/hostsim/liboracle_query.so: tests/hostsim/oracle_query.cpp oracle/oracle.cpp include/rtcuda.h
	g++ -O2 -std=c++17 -fPIC -ffp-contract=off -fno-fast-math -Wall -Wno-unused-function -pthread -shared -o $@ $<

# radiance along caller-supplied rays on the CPU (includes hostsim.cpp)
tests/hostsim/libhostsim_radiance.so: tests/hostsim/hostsim_radiance.cpp tests/hostsim/hostsim.cpp $(HDRS)
	g++ -O2 -std=c++17 -fPIC -shared -pthread -o $@ $<

# its reference: the oracle's ray_radiance per caller-supplied ray (includes oracle/oracle.cpp, built with the oracle's flags)
tests/hostsim/liboracle_radiance.so: tests/hostsim/oracle_radiance.cpp oracle/oracle.cpp include/rtcuda.h
	g++ -O2 -std=c++17 -fPIC -ffp-contract=off -fno-fast-math -Wall -Wno-unused-function -pthread -shared -o $@ $<

# the surface query on the CPU (includes hostsim.cpp)
tests/hostsim/libhostsim_surfaces.so: tests/hostsim/hostsim_surfaces.cpp tests/hostsim/hostsim.cpp $(HDRS)
	g++ -O2 -std=c++17 -fPIC -shared -pthread -o $@ $<

# its reference: the oracle's traverse_bvh HitInfo and get_albedo per caller-supplied ray (includes oracle/oracle.cpp, built with the
# oracle's flags)
tests/hostsim/liboracle_surfaces.so: tests/hostsim/oracle_surfaces.cpp oracle/oracle.cpp include/rtcuda.h
	g++ -O2 -std=c++17 -fPIC -ffp-contract=off -fno-fast-math -Wall -Wno-unused-function -pthread -shared -o $@ $<

clean:
	rm -rf build $(PKG)/libraytracing_cuda.so oracle/liboracle.so tests/hostsim/libhostsim.so tests/hostsim/libhostsim_update.so \
		tests/hostsim/libhostsim_query.so tests/hostsim/liboracle_query.so tests/hostsim/libhostsim_radiance.so tests/hostsim/liboracle_radiance.so \
		tests/hostsim/libhostsim_surfaces.so tests/hostsim/liboracle_surfaces.so
