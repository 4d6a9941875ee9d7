/* TEST INFRASTRUCTURE ONLY (see oracle/README.md).
 *
 * mdct_backward of libvorbis 1.3 (lib/mdct.c: mdct_init, the butterflies, mdct_bitreverse), float, transcribed with its
 * operation order kept. The reference's src/mdct.cpp is this code (its mdct_lookup is libvorbis'), and this transcription
 * reproduces every transform recorded in the reference's dumps under tests/golden bit for bit
 * (tests/test_oracle_golden.py), so the tests use it where they need the reference's transform on other inputs.
 *
 * The libvorbis code carries this notice:
 *
 * Copyright (c) 2002-2020 Xiph.org Foundation
 *
 * Redistribution and use in source and binary forms, with or without
 * modification, are permitted provided that the following conditions
 * are met:
 *
 * - Redistributions of source code must retain the above copyright
 * notice, this list of conditions and the following disclaimer.
 *
 * - Redistributions in binary form must reproduce the above copyright
 * notice, this list of conditions and the following disclaimer in the
 * documentation and/or other materials provided with the distribution.
 *
 * - Neither the name of the Xiph.org Foundation nor the names of its
 * contributors may be used to endorse or promote products derived from
 * this software without specific prior written permission.
 *
 * THIS SOFTWARE IS PROVIDED BY THE COPYRIGHT HOLDERS AND CONTRIBUTORS
 * ``AS IS'' AND ANY EXPRESS OR IMPLIED WARRANTIES, INCLUDING, BUT NOT
 * LIMITED TO, THE IMPLIED WARRANTIES OF MERCHANTABILITY AND FITNESS FOR
 * A PARTICULAR PURPOSE ARE DISCLAIMED.  IN NO EVENT SHALL THE FOUNDATION
 * OR CONTRIBUTORS BE LIABLE FOR ANY DIRECT, INDIRECT, INCIDENTAL,
 * SPECIAL, EXEMPLARY, OR CONSEQUENTIAL DAMAGES (INCLUDING, BUT NOT
 * LIMITED TO, PROCUREMENT OF SUBSTITUTE GOODS OR SERVICES; LOSS OF USE,
 * DATA, OR PROFITS; OR BUSINESS INTERRUPTION) HOWEVER CAUSED AND ON ANY
 * THEORY OF LIABILITY, WHETHER IN CONTRACT, STRICT LIABILITY, OR TORT
 * (INCLUDING NEGLIGENCE OR OTHERWISE) ARISING IN ANY WAY OUT OF THE USE
 * OF THIS SOFTWARE, EVEN IF ADVISED OF THE POSSIBILITY OF SUCH DAMAGE.
 */
#include <math.h>
#include <stdlib.h>
#ifndef M_PI
#define M_PI 3.14159265358979323846
#endif
#define cPI3_8 (.38268343236508977175F)
#define cPI2_8 (.70710678118654752441F)
#define cPI1_8 (.92387953251128675613F)
typedef struct { int n; int log2n; float *trig; int *bitrev; float scale; } mdct_lookup;

static void mdct_init(mdct_lookup *lookup, int n){
  int *bitrev = malloc(sizeof(*bitrev) * (n / 4));
  float *T = malloc(sizeof(*T) * (n + n / 4));
  int i, n2 = n >> 1;
  int log2n = lookup->log2n = rint(log((float) n) / log(2.f));
  lookup->n = n; lookup->trig = T; lookup->bitrev = bitrev;
  for(i = 0; i < n / 4; i++){
    T[i*2] = cos((M_PI/n)*(4*i));
    T[i*2+1] = -sin((M_PI/n)*(4*i));
    T[n2+i*2] = cos((M_PI/(2*n))*(2*i+1));
    T[n2+i*2+1] = sin((M_PI/(2*n))*(2*i+1));
  }
  for(i = 0; i < n / 8; i++){
    T[n+i*2] = cos((M_PI/n)*(4*i+2))*.5;
    T[n+i*2+1] = -sin((M_PI/n)*(4*i+2))*.5;
  }
  {
    int mask = (1 << (log2n - 1)) - 1, j;
    int msb = 1 << (log2n - 2);
    for(i = 0; i < n / 8; i++){
      int acc = 0;
      for(j = 0; msb >> j; j++)
        if((msb >> j) & i) acc |= 1 << j;
      bitrev[i*2] = ((~acc) & mask) - 1;
      bitrev[i*2+1] = acc;
    }
  }
  lookup->scale = 4.f / n;
}

static void mdct_butterfly_8(float *x){
  float r0 = x[6] + x[2];
  float r1 = x[6] - x[2];
  float r2 = x[4] + x[0];
  float r3 = x[4] - x[0];
  x[6] = r0 + r2;
  x[4] = r0 - r2;
  r0 = x[5] - x[1];
  r2 = x[7] - x[3];
  x[0] = r1 + r0;
  x[2] = r1 - r0;
  r0 = x[5] + x[1];
  r1 = x[7] + x[3];
  x[3] = r2 + r3;
  x[1] = r2 - r3;
  x[7] = r1 + r0;
  x[5] = r1 - r0;
}

static void mdct_butterfly_16(float *x){
  float r0 = x[1] - x[9];
  float r1 = x[0] - x[8];
  x[8] += x[0];
  x[9] += x[1];
  x[0] = ((r0 + r1) * cPI2_8);
  x[1] = ((r0 - r1) * cPI2_8);
  r0 = x[3] - x[11];
  r1 = x[10] - x[2];
  x[10] += x[2];
  x[11] += x[3];
  x[2] = r0;
  x[3] = r1;
  r0 = x[12] - x[4];
  r1 = x[13] - x[5];
  x[12] += x[4];
  x[13] += x[5];
  x[4] = ((r0 - r1) * cPI2_8);
  x[5] = ((r0 + r1) * cPI2_8);
  r0 = x[14] - x[6];
  r1 = x[15] - x[7];
  x[14] += x[6];
  x[15] += x[7];
  x[6] = r0;
  x[7] = r1;
  mdct_butterfly_8(x);
  mdct_butterfly_8(x + 8);
}

static void mdct_butterfly_32(float *x){
  float r0 = x[30] - x[14];
  float r1 = x[31] - x[15];
  x[30] += x[14];
  x[31] += x[15];
  x[14] = r0;
  x[15] = r1;
  r0 = x[28] - x[12];
  r1 = x[29] - x[13];
  x[28] += x[12];
  x[29] += x[13];
  x[12] = (r0 * cPI1_8 - r1 * cPI3_8);
  x[13] = (r0 * cPI3_8 + r1 * cPI1_8);
  r0 = x[26] - x[10];
  r1 = x[27] - x[11];
  x[26] += x[10];
  x[27] += x[11];
  x[10] = ((r0 - r1) * cPI2_8);
  x[11] = ((r0 + r1) * cPI2_8);
  r0 = x[24] - x[8];
  r1 = x[25] - x[9];
  x[24] += x[8];
  x[25] += x[9];
  x[8] = (r0 * cPI3_8 - r1 * cPI1_8);
  x[9] = (r1 * cPI3_8 + r0 * cPI1_8);
  r0 = x[22] - x[6];
  r1 = x[7] - x[23];
  x[22] += x[6];
  x[23] += x[7];
  x[6] = r1;
  x[7] = r0;
  r0 = x[4] - x[20];
  r1 = x[5] - x[21];
  x[20] += x[4];
  x[21] += x[5];
  x[4] = (r1 * cPI1_8 + r0 * cPI3_8);
  x[5] = (r1 * cPI3_8 - r0 * cPI1_8);
  r0 = x[2] - x[18];
  r1 = x[3] - x[19];
  x[18] += x[2];
  x[19] += x[3];
  x[2] = ((r1 + r0) * cPI2_8);
  x[3] = ((r1 - r0) * cPI2_8);
  r0 = x[0] - x[16];
  r1 = x[1] - x[17];
  x[16] += x[0];
  x[17] += x[1];
  x[0] = (r1 * cPI3_8 + r0 * cPI1_8);
  x[1] = (r1 * cPI1_8 - r0 * cPI3_8);
  mdct_butterfly_16(x);
  mdct_butterfly_16(x + 16);
}

#define BF_STEP(a, b, t0, t1) \
  r0 = x1[a] - x2[a]; r1 = x1[b] - x2[b]; x1[a] += x2[a]; x1[b] += x2[b]; \
  x2[a] = (r1 * (t1) + r0 * (t0)); x2[b] = (r1 * (t0) - r0 * (t1));

static void mdct_butterfly_first(float *T, float *x, int points){
  float *x1 = x + points - 8;
  float *x2 = x + (points >> 1) - 8;
  float r0, r1;
  do{
    BF_STEP(6, 7, T[0], T[1]);
    BF_STEP(4, 5, T[4], T[5]);
    BF_STEP(2, 3, T[8], T[9]);
    BF_STEP(0, 1, T[12], T[13]);
    x1 -= 8; x2 -= 8; T += 16;
  }while(x2 >= x);
}

static void mdct_butterfly_generic(float *T, float *x, int points, int trigint){
  float *x1 = x + points - 8;
  float *x2 = x + (points >> 1) - 8;
  float r0, r1;
  do{
    BF_STEP(6, 7, T[0], T[1]); T += trigint;
    BF_STEP(4, 5, T[0], T[1]); T += trigint;
    BF_STEP(2, 3, T[0], T[1]); T += trigint;
    BF_STEP(0, 1, T[0], T[1]); T += trigint;
    x1 -= 8; x2 -= 8;
  }while(x2 >= x);
}

static void mdct_butterflies(mdct_lookup *init, float *x, int points){
  float *T = init->trig;
  int stages = init->log2n - 5;
  int i, j;
  if(--stages > 0) mdct_butterfly_first(T, x, points);
  for(i = 1; --stages > 0; i++)
    for(j = 0; j < (1 << i); j++)
      mdct_butterfly_generic(T, x + (points >> i) * j, points >> i, 4 << i);
  for(j = 0; j < points; j += 32) mdct_butterfly_32(x + j);
}

static void mdct_bitreverse(mdct_lookup *init, float *x){
  int n = init->n;
  int *bit = init->bitrev;
  float *w0 = x;
  float *w1 = x = w0 + (n >> 1);
  float *T = init->trig + n;
  do{
    float *x0 = x + bit[0];
    float *x1 = x + bit[1];
    float r0 = x0[1] - x1[1];
    float r1 = x0[0] + x1[0];
    float r2 = (r1 * T[0] + r0 * T[1]);
    float r3 = (r1 * T[1] - r0 * T[0]);
    w1 -= 4;
    r0 = (x0[1] + x1[1]) * .5f;
    r1 = (x0[0] - x1[0]) * .5f;
    w0[0] = r0 + r2;
    w1[2] = r0 - r2;
    w0[1] = r1 + r3;
    w1[3] = r3 - r1;
    x0 = x + bit[2];
    x1 = x + bit[3];
    r0 = x0[1] - x1[1];
    r1 = x0[0] + x1[0];
    r2 = (r1 * T[2] + r0 * T[3]);
    r3 = (r1 * T[3] - r0 * T[2]);
    r0 = (x0[1] + x1[1]) * .5f;
    r1 = (x0[0] - x1[0]) * .5f;
    w0[2] = r0 + r2;
    w1[0] = r0 - r2;
    w0[3] = r1 + r3;
    w1[1] = r3 - r1;
    T += 4; bit += 4; w0 += 4;
  }while(w0 < w1);
}

/* out[n] = mdct_backward(in[n/2]), n a power of two from 64 to 8192 */
void por_vorbis_mdct_backward(int n, const float *in, float *out){
  mdct_lookup L; mdct_lookup *init = &L;
  mdct_init(init, n);
  int n2 = n >> 1, n4 = n >> 2;
  const float *iX = in + n2 - 7;
  float *oX = out + n2 + n4;
  float *T = init->trig + n4;
  do{
    oX -= 4;
    oX[0] = (-iX[2] * T[3] - iX[0] * T[2]);
    oX[1] = (iX[0] * T[3] - iX[2] * T[2]);
    oX[2] = (-iX[6] * T[1] - iX[4] * T[0]);
    oX[3] = (iX[4] * T[1] - iX[6] * T[0]);
    iX -= 8; T += 4;
  }while(iX >= in);
  iX = in + n2 - 8;
  oX = out + n2 + n4;
  T = init->trig + n4;
  do{
    T -= 4;
    oX[0] = (iX[4] * T[3] + iX[6] * T[2]);
    oX[1] = (iX[4] * T[2] - iX[6] * T[3]);
    oX[2] = (iX[0] * T[1] + iX[2] * T[0]);
    oX[3] = (iX[0] * T[0] - iX[2] * T[1]);
    iX -= 8; oX += 4;
  }while(iX >= in);
  mdct_butterflies(init, out + n2, n2);
  mdct_bitreverse(init, out);
  {
    float *oX1 = out + n2 + n4, *oX2 = out + n2 + n4, *iX = out;
    T = init->trig + n2;
    do{
      oX1 -= 4;
      oX1[3] = (iX[0] * T[1] - iX[1] * T[0]);
      oX2[0] = -(iX[0] * T[0] + iX[1] * T[1]);
      oX1[2] = (iX[2] * T[3] - iX[3] * T[2]);
      oX2[1] = -(iX[2] * T[2] + iX[3] * T[3]);
      oX1[1] = (iX[4] * T[5] - iX[5] * T[4]);
      oX2[2] = -(iX[4] * T[4] + iX[5] * T[5]);
      oX1[0] = (iX[6] * T[7] - iX[7] * T[6]);
      oX2[3] = -(iX[6] * T[6] + iX[7] * T[7]);
      oX2 += 4; iX += 8; T += 8;
    }while(iX < oX1);
    iX = out + n2 + n4; oX1 = out + n4; oX2 = oX1;
    do{
      oX1 -= 4; iX -= 4;
      oX2[0] = -(oX1[3] = iX[3]);
      oX2[1] = -(oX1[2] = iX[2]);
      oX2[2] = -(oX1[1] = iX[1]);
      oX2[3] = -(oX1[0] = iX[0]);
      oX2 += 4;
    }while(oX2 < iX);
    iX = out + n2 + n4; oX1 = out + n2 + n4; oX2 = out + n2;
    do{
      oX1 -= 4;
      oX1[0] = iX[3]; oX1[1] = iX[2]; oX1[2] = iX[1]; oX1[3] = iX[0];
      iX += 4;
    }while(oX1 > oX2);
  }
  free(init->trig); free(init->bitrev);
}
