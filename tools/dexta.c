/* dexta -- .fasta -> .dexta (2 bits per base).
 * Same command line, flags and file format as the reference's dexta (dexta.c:19-66); the work is
 * done by libdexb200.so on the GPU (see dxcli.h). */
#include "dxcli.h"

static int run(dx_ctx *ctx, const dx_opts *o, const uint8_t *d_in, size_t n,
               uint8_t **d_out, size_t *out_len)
{ size_t cap = n/3 + 200000;            /* the usual case; an image has no a-priori bound (17 bytes per
                                          entry, 0xff bytes for well gaps): ask again with what it needs */
  int rc = DX_OK;
  (void) o;
  for (int attempt = 0; attempt < 2; attempt++)
    { *d_out = (uint8_t *) dx_device_alloc(ctx,cap);
      if (*d_out == NULL) return DX_E_NOMEM;
      rc = dx_dexta_dev(ctx,DX_FASTA,d_in,n,*d_out,cap,out_len);
      if (rc != DX_E_CAP || dx_needed_bytes(ctx) <= cap) break;
      dx_device_free(ctx,*d_out); *d_out = NULL;
      cap = dx_needed_bytes(ctx) + 64;
    }
  return rc;
}

static int stream(dx_win *w) { return dx_stream_pack(w,DX_FASTA); }

int main(int argc, char *argv[])
{ static const dx_tool tool =
    { "dexta", "[-vk] ( -i | <path:fasta> ... )", "vki", 0, ".fasta", ".dexta",
      { "      -i: source is on standard input.",
        "      -k: do *not* remove the .fasta file on completion.",
        "      -w: line width for sequence lines.", NULL, NULL }, run, stream, 4.0 };
  return dx_cli_main(&tool,argc,argv);
}
