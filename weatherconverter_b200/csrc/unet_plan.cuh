// The UNet's topology (diffusion_model/models/unet_base.py:372-488), shared by the inference plan (unet.cu) and the
// training plan (unet_train.cu): config checks, the t_emb_layers table and the down / mid / up walk.  Each plan supplies a
// builder with the layer hooks and keeps its own preamble (time embedding) and head (norm_out + conv_out).
//
// Skip connections are written by their producers directly into the second half of the up-path concat buffers, and the
// up-sampling transposed conv writes the first half (unet_base.py:348-349), so torch.cat never runs.
#pragma once
#include <string>
#include <utility>
#include <vector>

#include "plan.cuh"
#include "../../include/wc_b200.h"

namespace wc {

inline int check_unet_config(const wc_unet_config& c) {
  WC_REQUIRE(c.im_channels == 3, "UNet boundary kernels support im_channels == 3");
  WC_REQUIRE(c.n_down_channels >= 2 && c.n_down_channels <= 8 && c.n_mid_channels >= 2, "bad channel lists");
  for (int i = 0; i < c.n_down_channels; ++i) WC_REQUIRE(c.down_channels[i] % 64 == 0, "channels must be multiples of 64");
  for (int i = 0; i < c.n_mid_channels; ++i) WC_REQUIRE(c.mid_channels[i] % 64 == 0, "channels must be multiples of 64");
  return 0;
}

inline int check_unet_hw(const wc_unet_config& c, int H, int W) {
  int div = 1;
  for (int i = 0; i + 1 < c.n_down_channels; ++i) if (c.down_sample[i]) div *= 2;
  WC_REQUIRE(H % div == 0 && W % div == 0, "H and W must be divisible by the total down-sampling factor");
  return 0;
}

// Every t_emb_layers Linear (unet_base.py:96-98) in execution order: (name prefix, output channels).  The plans
// concatenate them so that one launch projects them all.
inline std::vector<std::pair<std::string, int>> temb_layers(const wc_unet_config& c) {
  const int nlev = c.n_down_channels - 1;
  const int* dc = c.down_channels;
  std::vector<std::pair<std::string, int>> tl;
  for (int i = 0; i < nlev; ++i)
    for (int l = 0; l < c.num_down_layers; ++l)
      tl.push_back({"downs." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", dc[i + 1]});
  for (int i = 0; i + 1 < c.n_mid_channels; ++i)
    for (int l = 0; l < c.num_mid_layers + 1; ++l)
      tl.push_back({"mids." + std::to_string(i) + ".t_emb_layers." + std::to_string(l) + ".1", c.mid_channels[i + 1]});
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    for (int l = 0; l < c.num_up_layers; ++l)
      tl.push_back({"ups." + std::to_string(j) + ".t_emb_layers." + std::to_string(l) + ".1", i != 0 ? dc[i - 1] : dc[0]});
  }
  return tl;
}

inline bool use_attn(const wc_unet_config& c, int level) {
  const int res = c.im_size >> level;
  for (int k = 0; k < c.n_attn_resolutions; ++k)
    if (c.attn_resolutions[k] == res) return true;
  return false;
}

// Allocates the concat buffers and walks conv_in, the down, mid and up paths through the builder's hooks
//   conv_in(skip0), resnet(x, cout, prefix, layer, dest), attention(x, prefix, layer, heads, dest),
//   down_sample(x, prefix, channels, out), up_sample(x, prefix, channels, out)
// (dest: where the layer writes its output, or nullptr for a fresh buffer).  Returns the activation norm_out reads; on
// failure b.err is set.
template <class Builder>
Act walk_unet(Builder& b, const wc_unet_config& c, int H, int W) {
  const int nlev = c.n_down_channels - 1;
  const int* dc = c.down_channels;

  // ---- level geometry and concat buffers
  std::vector<int> LH(nlev + 1), LW(nlev + 1);
  LH[0] = H; LW[0] = W;
  for (int i = 0; i < nlev; ++i) {
    LH[i + 1] = c.down_sample[i] ? LH[i] / 2 : LH[i];
    LW[i + 1] = c.down_sample[i] ? LW[i] / 2 : LW[i];
  }
  std::vector<Act> cat(nlev);
  for (int i = 0; i < nlev; ++i) cat[i] = b.act(LH[i], LW[i], 2 * dc[i]);

  // ---- conv_in, written straight into the level-0 skip slot
  Act skip0 = slice_act(cat[0], dc[0], dc[0]);
  b.conv_in(skip0);
  Act cur = skip0;

  // ---- down path (unet_base.py:466-468, DownBlock.forward :131-164)
  for (int i = 0; i < nlev; ++i) {
    const std::string p = "downs." + std::to_string(i);
    const bool ua = use_attn(c, i);
    // The block output is the skip of level i+1 (if it exists); route it into that concat buffer.
    const bool has_next_skip = (i + 1 != nlev);
    Act next_skip;
    if (has_next_skip) next_skip = slice_act(cat[i + 1], dc[i + 1], dc[i + 1]);
    for (int l = 0; l < c.num_down_layers; ++l) {
      const bool final_op = (l + 1 == c.num_down_layers) && !c.down_sample[i] && has_next_skip;
      cur = b.resnet(cur, dc[i + 1], p, l, (final_op && !ua) ? &next_skip : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &next_skip : nullptr);
    }
    if (c.down_sample[i]) {
      Act out = has_next_skip ? next_skip : b.act(LH[i + 1], LW[i + 1], dc[i + 1]);
      b.down_sample(cur, p, dc[i + 1], out);
      cur = out;
    }
    if (b.err) return cur;
  }

  // ---- mid blocks (MidBlock.forward :228-268)
  for (int i = 0; i + 1 < c.n_mid_channels; ++i) {
    const std::string p = "mids." + std::to_string(i);
    const int cout = c.mid_channels[i + 1];
    // The last mid output feeds the first up block; if that block does not up-sample it is the first half of its
    // concat buffer.
    const int top = nlev - 1;
    const bool direct = (i + 2 == c.n_mid_channels) && !c.down_sample[top];
    Act dest = slice_act(cat[top], 0, dc[top]);
    cur = b.resnet(cur, cout, p, 0, nullptr);
    for (int l = 0; l < c.num_mid_layers; ++l) {
      cur = b.attention(cur, p, l, c.num_heads, nullptr);
      const bool final_op = direct && (l + 1 == c.num_mid_layers);
      cur = b.resnet(cur, cout, p, l + 1, final_op ? &dest : nullptr);
    }
    if (b.err) return cur;
  }

  // ---- up path (UpBlock.forward :336-369)
  for (int j = 0; j < nlev; ++j) {
    const int i = nlev - 1 - j;
    const std::string p = "ups." + std::to_string(j);
    const bool ua = use_attn(c, i);
    const int cout = i != 0 ? dc[i - 1] : dc[0];
    Act first_half = slice_act(cat[i], 0, dc[i]);
    if (c.down_sample[i]) {
      b.up_sample(cur, p, dc[i], first_half);
      if (b.err) return cur;
    } else if (cur.ptr != first_half.ptr) {
      b.err = fail("internal: up block without up-sampling expects its input inside the concat buffer");
      return cur;
    }
    cur = cat[i];
    // If the next (finer) up block does not up-sample, this block's output is the first half of its concat buffer.
    const bool direct = (i > 0) && !c.down_sample[i - 1];
    Act dest = direct ? slice_act(cat[i - 1], 0, dc[i - 1]) : Act();
    for (int l = 0; l < c.num_up_layers; ++l) {
      const bool final_op = direct && (l + 1 == c.num_up_layers);
      cur = b.resnet(cur, cout, p, l, (final_op && !ua) ? &dest : nullptr);
      if (ua) cur = b.attention(cur, p, l, c.num_heads, final_op ? &dest : nullptr);
    }
    if (b.err) return cur;
  }
  return cur;
}

}  // namespace wc
