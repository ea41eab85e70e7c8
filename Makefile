# Builds the C-ABI kernel library (sm_100a only): stable-video-infinity_b200/lib/libsvi_b200.so
NVCC ?= nvcc
PKG := stable-video-infinity_b200
CSRC := $(PKG)/csrc
LIB := $(PKG)/lib/libsvi_b200.so
NVFLAGS := -gencode arch=compute_100a,code=sm_100a -O3 -lineinfo -std=c++17 -Xcompiler -fPIC
SRCS := $(CSRC)/runtime.cu $(CSRC)/gemm_tcgen05.cu $(CSRC)/gemm2_tcgen05.cu $(CSRC)/attn_tcgen05.cu $(CSRC)/sp_exchange.cu $(CSRC)/elementwise.cu $(CSRC)/conv3d_tcgen05.cu $(CSRC)/conv3d2_tcgen05.cu $(CSRC)/vae_elementwise.cu $(CSRC)/encoder_kernels.cu $(CSRC)/audio_kernels.cu
OBJS := $(patsubst $(CSRC)/%.cu,build/%.o,$(SRCS))

all: $(LIB)

build/%.o: $(CSRC)/%.cu $(CSRC)/common.cuh $(CSRC)/conv3d_common.cuh $(CSRC)/gemm_epilogue.cuh include/svi_b200.h
	@mkdir -p build
	$(NVCC) $(NVFLAGS) -Xptxas -v -c $< -o $@ 2> build/$*.ptxas.log || (cat build/$*.ptxas.log; exit 1)

$(LIB): $(OBJS)
	@mkdir -p $(PKG)/lib
	$(NVCC) -shared -o $@ $(OBJS) -cudart shared

# experimental kernels (csrc/experimental/README.md): a separate library, never loaded by the package
EXP_LIB := $(PKG)/lib/libsvi_b200_exp.so
EXP_SRCS := $(CSRC)/runtime.cu $(CSRC)/experimental/attn4_tcgen05.cu $(CSRC)/experimental/exp_entry.cu
exp:
	@mkdir -p $(PKG)/lib build
	$(NVCC) $(NVFLAGS) -shared -o $(EXP_LIB) $(EXP_SRCS) -cudart shared

# A/B build with --use_fast_math (measurement only: SVI_B200_LIB=<this file> selects it; never the default)
FM_LIB := $(PKG)/lib/libsvi_b200_fastmath.so
fastmath:
	@mkdir -p $(PKG)/lib build
	$(NVCC) $(NVFLAGS) --use_fast_math -shared -o $(FM_LIB) $(SRCS) -cudart shared

# attention A/B builds (measurement only, selected with SVI_B200_LIB): share of exponentials on the FMA-pipe polynomial
attn_variants:
	@mkdir -p $(PKG)/lib build
	$(NVCC) $(NVFLAGS) -DSVI_ATTN_COLSPLIT=1 -shared -o $(PKG)/lib/libsvi_b200_attn_colsplit.so $(SRCS) -cudart shared
	$(NVCC) $(NVFLAGS) -DSVI_ATTN_COLSPLIT=1 -DSVI_ATTN_POLY16=4 -shared -o $(PKG)/lib/libsvi_b200_attn_colsplit_p4.so $(SRCS) -cudart shared
	$(NVCC) $(NVFLAGS) -DSVI_ATTN_COLSPLIT=1 -DSVI_ATTN_POLY16=7 -shared -o $(PKG)/lib/libsvi_b200_attn_colsplit_p7.so $(SRCS) -cudart shared
	$(NVCC) $(NVFLAGS) -DSVI_ATTN_COLSPLIT=1 -DSVI_ATTN_OTHER_REGS=120 -DSVI_ATTN_SOFTMAX_REGS=192 -shared -o $(PKG)/lib/libsvi_b200_attn_colsplit_r192.so $(SRCS) -cudart shared

# the library with the ROUND-1 attention kernel (320 threads, 168 registers, 6/16 polynomial share) for same-box A/B runs
attn_r1:
	@mkdir -p $(PKG)/lib build
	$(NVCC) $(NVFLAGS) -shared -o $(PKG)/lib/libsvi_b200_attn_r1.so $(filter-out $(CSRC)/attn_tcgen05.cu,$(SRCS)) $(CSRC)/experimental/attn_r1_tcgen05.cu -cudart shared

clean:
	rm -rf build $(LIB) $(EXP_LIB)
.PHONY: all clean exp fastmath attn_variants attn_r1

# A/B builds of the pair convolution kernel (SVI_B200_LIB=<lib> python tools/gpu_check.py perf_conv): u = uniform MMA operands,
# e = epilogue that keeps the result in registers and frees the accumulator after the first pass
CONV_OTHER := $(filter-out build/conv3d2_tcgen05.o,$(OBJS))
conv_variants: $(OBJS)
	for v in u0e1 u1e0 u0e0; do \
	  u=$$(echo $$v | cut -c2); e=$$(echo $$v | cut -c4); \
	  $(NVCC) $(NVFLAGS) -DSVI_CONV2_UNIFORM=$$u -DSVI_CONV2_EPI=$$e -c $(CSRC)/conv3d2_tcgen05.cu -o build/conv3d2_$$v.o && \
	  $(NVCC) -shared -o $(PKG)/lib/libsvi_b200_conv_$$v.so $(CONV_OTHER) build/conv3d2_$$v.o -cudart shared || exit 1; \
	done
